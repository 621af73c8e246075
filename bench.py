#!/usr/bin/env python3
"""bench.py -- megapixels/sec of the stage 01-03 hot path (resize + colour layers + edges) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload config5|config2|config3|config4]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one image per GPU: 01 resize_if_needed (a no-op for the
named config, exactly as in the reference: max_dimension = image size), 02 nearest-centre assignment
in 8-bit Lab -> K layer masks (+RECT-3 open/close), 03 per-layer ELLIPSE-3 open/close -> Gaussian blur
-> Canny.  K-means centres are an INPUT of the path (computed once on the host before timing, the way
02_color_extract.py:39-49 does) for both arms.

  workload   default = the shape north_star quotes its target on (BASELINE configs[4] image: 4096x4096, 16 colours, Canny
             50/150, blur 3); configs[1] and configs[2] are measured in the same run as extra records (N = 1), configs[3]
             (512 x 1080p frames sharded over the ranks, strong scaling) as the `configs3` record at every N.
  value      device-resident: image already in HBM, masks+edges (u8 planes) left in HBM; CUDA events per step on
             the launching stream, L2 flushed (untimed) between steps; max over ranks.  Single-image workloads rebuild the
             candidate-centre tables every step (a new image has new k-means centres).
  e2e        the same through the host-buffer C-ABI call with pinned host buffers, every step: omni_host_color_edge_packed
             (image in, the K masks and K edge planes out as 1 bit per pixel -- what the drop-in stage scripts write into
             1-bit PNGs); `e2e_u8` is the byte-plane call omni_host_color_edge.
  roofline   dominant kernel of the step, CUDA-event timed inside the timed region (omni_profile_*).
  cpu_baseline / --impl reference
             the reference's own CPU implementation of the path (oracle/refport.py: the cv2/NumPy call
             sites of 02:35-36,53-55,121-154 and 03:23-34 replayed verbatim; /root/reference is Python
             and cannot travel to the GPU box), timed on this box's host cores.

N > 1: launched by torchrun, one rank per GPU, frames sharded by rank (weak scaling, no data-path
collective; torch.distributed is used only for the barrier and the max-over-ranks of the timing).
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "omnirevolve-image-processor_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

WORKLOADS = {
    "config2": dict(h=4096, w=4096, K=8, seed=0, cell=32, low=50, high=150, ksize=3,
                    name="configs[1]: single 4096x4096 RGB image, 8 colours, Canny 50/150, blur 3, max_dimension=4096"),
    "config3": dict(h=8192, w=8192, K=16, seed=1, cell=64, low=50, high=150, ksize=3,
                    name="configs[2]: single 8192x8192 image, 16 colours, per-layer edge masks"),
    "config4": dict(h=1080, w=1920, K=8, seed=0, cell=32, low=50, high=150, ksize=3, batch=4,
                    name="configs[3]: 1920x1080 frames, 8 colours, one centre set; a step = 4 frames per GPU through omni_color_edge_batch"),
    # BASELINE.json configs[4] at its default Canny point = the north-star's "4Kx4K, 16 colours" target shape
    "config5": dict(h=4096, w=4096, K=16, seed=0, cell=32, low=50, high=150, ksize=3,
                    name="configs[4] image: 4096x4096, 16 colours, Canny 50/150, blur 3 (the north-star target shape)"),
    "small": dict(h=1024, w=1024, K=4, seed=0, cell=32, low=50, high=150, ksize=3,
                  name="configs[0] shape: 1024x1024, 4 colours"),
}
METRIC = "megapixels/sec (resize+color+edge)"
UNIT = "MP/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz, self.err = index, [], set(), False, None, None
        self.power = []

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
                if len(self.samples) % 4 == 1:                 # (every NVML query is a round trip to the GPU's management unit)
                    try:
                        self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    except Exception:
                        pass
                time.sleep(0.010)
        except Exception as exc:                       # noqa: BLE001
            self.err = repr(exc)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "error": self.err}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "power_w_max": max(self.power) if self.power else None}


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's cv2 + NumPy call sites, timed on the host
# ------------------------------------------------------------------------------------------------------
def cpu_path_once(rp, img, centers, K, wl):
    """02:35-36,53-55 assign -> :121-127 relabel -> :146-154 masks -> 03:23-34 edges, in-process, no PNG I/O."""
    labels = rp.assign_lab(img, centers)
    _order, lut = rp.darkness_order(centers)
    masks = rp.layer_masks(lut[labels], K)
    edges = rp.edges_all(masks, low=wl["low"], high=wl["high"], ksize=wl["ksize"])
    return masks, edges


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import cv2
    from oracle import refport as rp
    from omni_b200.synth import synth
    img = synth(wl["h"], wl["w"], wl["seed"], wl["cell"])
    K = wl["K"]
    centers = rp.kmeans_lab_centers(img, K)
    # bounded sample per step: a band of rows sized for ~1 s of CPU work (the full image takes ~11 s at 4096^2, K=8)
    rows = max(64, min(wl["h"], int(2.0e6 // wl["w"])))
    band = np.ascontiguousarray(img[:rows])
    for _ in range(args.warmup):
        cpu_path_once(rp, band, centers, K, wl)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_path_once(rp, band, centers, K, wl)
    dt = time.perf_counter() - t0
    mp = rows * wl["w"] / 1e6
    val = mp * args.steps / dt
    cores = cv2.getNumThreads()
    sample = (f"{rows} rows x {wl['w']} px band of the {wl['h']}x{wl['w']} image per step ({mp:.2f} MP), K={K}; "
              f"NumPy assignment single-threaded as in the reference, OpenCV ops on {cores} threads; k-means centres precomputed")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": wl["name"], "K": K, "h": wl["h"], "w": wl["w"], "sample_rows": rows},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_baseline_leg(wl, img, centers):
    """Rank 0, N=1: the full reference CPU path on ONE full image of the workload (bounded: ~10-30 s)."""
    import cv2
    from oracle import refport as rp
    K = wl["K"]
    rows = wl["h"] if wl["h"] * wl["w"] * K <= 4096 * 4096 * 8 else max(64, int(4096 * 4096 * 8 // (wl["w"] * K)))
    band = np.ascontiguousarray(img[:rows])
    t0 = time.perf_counter()
    cpu_path_once(rp, band, centers, K, wl)
    dt = time.perf_counter() - t0
    mp = rows * wl["w"] / 1e6
    return {"value": mp / dt, "unit": UNIT, "cores": cv2.getNumThreads(), "kind": "port", "host_cpus": os.cpu_count(),
            "seconds": dt,
            "sample": (f"one pass over {rows}x{wl['w']} px ({mp:.1f} MP) of the workload image, K={K}: oracle/refport.py = the "
                       "reference's cv2/NumPy call sites (02:35-36,53-55,121-154; 03:23-34) in-process, no PNG I/O, "
                       "k-means centres precomputed; NumPy assignment single-threaded as in the reference")}


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
KERNEL_BYTES = {
    # algorithmic bytes per launch: the u8 image / mask / edge tensors a kernel must read or write in HBM
    # (N = H*W pixels, K planes; bit-plane intermediates count zero -- SURVEY 8d, DESIGN.md 4)
    "assign": lambda N, K: N * (3 + 1),
    "onehot": lambda N, K: N * (1 + K),
    "morph": lambda N, K: N * 2 * K,
    "blur": lambda N, K: N * 2 * K,
    "canny_nms": lambda N, K: N * 2 * K,
    "hyst_pass": lambda N, K: N * 2 * K,
    "hyst_final": lambda N, K: N * 2 * K,
    "assign_bits": lambda N, K: N * 3,               # image read; label bit-slices stay in L2
    "label_open": lambda N, K: 0,                    # bit-planes only
    "morph_bits": lambda N, K: N * K,                # mask byte planes written
    "edges3_bits": lambda N, K: N * K,               # bit-planes in; edge byte planes (strong set) written
    "hysteresis_bits": lambda N, K: 0,               # bit-planes only + a few promoted pixels
    "build_cells": lambda N, K: 0,
    "build_rgbcells": lambda N, K: 0,
    "build_tables": lambda N, K: 0,
}
# stage grouping for the report: colour = image -> K masks, edge = K masks -> K edges (masks are not re-read)
STAGES = {"color": ("build_cells", "build_rgbcells", "build_tables", "assign_bits", "label_open", "morph_bits", "assign", "onehot"),
          "edge": ("edge_runs", "edges3_bits", "hysteresis_bits", "morph", "blur", "canny_nms", "hyst_pass", "hyst_final")}


DUMP_BYTES = 64 * 10**6


def output_sample(torch, outs, seed=0):
    """--dump-outputs: the u8 planes a caller of the timed call receives, as float32 arrays.  An output that fits its share of
    DUMP_BYTES is kept whole; a larger one by its values at a fixed, seeded set of flat positions (the same for the same
    workload on every run), beside `<name>_nonzero`, the nonzero count of every plane of the whole output."""
    per = (DUMP_BYTES - 10**6) // 4 // len(outs)
    res = {}
    for name, t in outs.items():
        n = t.numel()
        if n <= per:
            res[name] = t.float().cpu().numpy()
        else:
            pos = np.unique(np.random.default_rng(seed).integers(0, n, per))
            res[name] = t.reshape(-1)[torch.from_numpy(pos).to(t.device)].float().cpu().numpy()
        res[name + "_nonzero"] = t.reshape(t.shape[:-2] + (-1,)).count_nonzero(-1).double().cpu().numpy()
    return res


def measure_fused(torch, eng, wl, img, centers, lut, steps, warmup, flush, barrier, cache_tables, dump=False):
    """Device-resident fused call on one image (or one frame batch): CUDA events per step, L2 flushed (untimed) between steps,
    then a second pass of the same steps with per-kernel events.  dump: also return device copies of the last timed step's outputs."""
    import omni_b200
    h, w, K = wl["h"], wl["w"], wl["K"]
    B = int(wl.get("batch", 1))
    ec = omni_b200.EdgeConfig(low=wl["low"], high=wl["high"], ksize=wl["ksize"])
    d_img = torch.from_numpy(img).cuda()
    d_masks = torch.empty(((B, K, h, w) if B > 1 else (K, h, w)), dtype=torch.uint8, device="cuda")
    d_edges = torch.empty_like(d_masks)
    eng.set_table_cache(cache_tables)

    def step():
        # 01: resize_if_needed is a no-op here (max_dimension == image size), as in the reference
        if B > 1:
            eng.color_edge_batch(d_img, centers, lut, ec, masks=d_masks, edges=d_edges)
        else:
            eng.color_edge(d_img, centers, lut, ec, masks=d_masks, edges=d_edges)

    for _ in range(max(warmup, 3)):
        step()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    n0 = eng.launch_count()
    barrier()
    t0 = time.perf_counter()
    for a, b in ev:
        flush.fill_(1)                       # L2 flush, outside the event-timed span
        a.record()
        step()
        b.record()
    barrier()
    wall = time.perf_counter() - t0
    launches = eng.launch_count() - n0
    last = {"masks": d_masks.clone(), "edges": d_edges.clone()} if dump else None
    eng.profile(True)
    pev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in pev:
        flush.fill_(1)
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    prof = eng.profile_summary()
    eng.profile(False)
    eng.set_table_cache(True)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    return {"step_ms": step_ms, "total_ms": sum(step_ms), "launches": launches, "prof": prof,
            "prof_step_ms": sum(a.elapsed_time(b) for a, b in pev) / steps, "wall": wall, "passes": eng.last_hysteresis_passes(),
            "d_edges": d_edges, "ec": ec, "last": last}


def roofline_record(prof, prof_step_ms, ms_per_step, steps, N, K, workload, peak, peak_src):
    dom = max(prof.items(), key=lambda kv: kv[1][1]) if prof else None
    if dom is None:
        return None
    name, (n_l, ms) = dom
    per_launch_ms = ms / n_l
    bytes_fn = KERNEL_BYTES.get(name)
    alg = bytes_fn(N * steps / n_l, K) if bytes_fn else None        # pixels per launch of this kernel
    ach = alg / (per_launch_ms / 1e3) / 1e9 if alg is not None else None
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get(workload, {}).get(name)
        except Exception:
            traffic = None
    step_bytes = N * (3 + 2 * K)
    return {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s",
            "frac": (ach / peak) if ach is not None else None, "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg, "launches_per_step": n_l / steps,
            "ms_per_launch": per_launch_ms, "share_of_step": ms / (prof_step_ms * steps),
            "timing": "CUDA events around every kernel launch, second pass of the same K steps (%.4f ms/step with the "
                      "events vs %.4f without)" % (prof_step_ms, ms_per_step),
            "step": {"algorithmic_bytes": step_bytes, "achieved": step_bytes / (ms_per_step / 1e3) / 1e9,
                     "frac": step_bytes / (ms_per_step / 1e3) / 1e9 / peak},
            "kernels_ms_per_step": {k: v[1] / steps for k, v in prof.items()},
            "kernels_frac_of_peak": {k: (KERNEL_BYTES[k](N * steps / v[0], K) / (v[1] / v[0] / 1e3) / 1e9 / peak)
                                     for k, v in prof.items() if k in KERNEL_BYTES and KERNEL_BYTES[k](N, K)},
            "stages_ms_per_step": {sname: sum(v[1] for k, v in prof.items() if k in members) / steps
                                   for sname, members in STAGES.items()},
            # what the dominant kernel itself moved through DRAM (ncu capture), over its live duration
            "achieved_from_traffic": (traffic / (per_launch_ms / 1e3) / 1e9) if traffic else None,
            "note": "edges3_bits walks only the live tile runs; the zeros of the dead tiles (the rest of its K*N algorithmic bytes) "
                    "are bulk copies (TMA engine) issued by assign_bits inside the timed step -- `step` is the figure that "
                    "accounts for everything"}


def configs3_record(torch, dist, eng, rank, world, flush, barrier, n_frames, peak):
    """BASELINE configs[3]: a batch of 1920x1080 frames, 8 colours, ONE centre set, sharded over the ranks in contiguous blocks
    (omni_b200/batch.py), strong scaling: every rank handles ceil(B / G) frames, no data-path collective.
    kernel: frames resident in HBM, u8 planes left in HBM (groups of 4 frames per omni_color_edge_batch call).
    e2e   : pinned host frames -> omni_host_color_edge_packed (H2D / kernels / D2H of consecutive groups overlapped) -> packed masks and
            edges in pinned host memory + per-frame counts, gathered to rank 0 in frame order."""
    import omni_b200
    from omni_b200 import batch as ob
    from omni_b200.synth import synth
    from omni_b200 import stages
    h, w, K = 1080, 1920, 8
    distinct = 16                                       # distinct synthetic frames, repeated to fill the batch
    base = [synth(h, w, 1000 + i, 32) for i in range(distinct)]
    centers = stages.kmeans_lab_centers(base[0], K)
    _o, lut = stages.darkness_lut(centers)
    lut = lut.astype(np.uint8)
    ec = omni_b200.EdgeConfig()
    mine = ob.shard_range(n_frames, world, rank)
    n_mine = len(mine)
    rb = (w + 7) // 8
    h_frames = omni_b200.pinned_empty((max(1, n_mine), h, w, 3))
    for j, f in enumerate(mine):
        h_frames[j] = base[f % distinct]
    h_mb = omni_b200.pinned_empty((max(1, n_mine) * K, h, rb))
    h_eb = omni_b200.pinned_empty((max(1, n_mine) * K, h, rb))
    # ---- kernel only ----
    G = 32 // K
    d_grp = torch.from_numpy(np.stack([base[i % distinct] for i in range(G)])).cuda()
    d_m = torch.empty((G, K, h, w), dtype=torch.uint8, device="cuda")
    d_e = torch.empty_like(d_m)
    for _ in range(3):
        eng.color_edge_batch(d_grp, centers, lut, ec, masks=d_m, edges=d_e)
    n_calls = (n_mine + G - 1) // G
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n_calls):
        eng.color_edge_batch(d_grp, centers, lut, ec, masks=d_m, edges=d_e)
    b.record()
    barrier()
    k_ms = a.elapsed_time(b) if n_calls else 0.0
    # ---- e2e ----
    if n_mine:
        eng.host_color_edge_packed(h_frames[:min(n_mine, 2 * G)], centers, lut, ec, mask_bits=h_mb[:min(n_mine, 2 * G) * K],
                                   edge_bits=h_eb[:min(n_mine, 2 * G) * K], want_counts=False)
    barrier()
    t0 = time.perf_counter()
    counts, _r = ob.process_shard_packed(eng, h_frames, mine, centers, lut, ec, mask_bits=h_mb[:n_mine * K] if n_mine else None,
                                         edge_bits=h_eb[:n_mine * K] if n_mine else None)
    torch.cuda.synchronize()
    e_s = time.perf_counter() - t0
    barrier()
    allc = ob.gather_counts(counts, n_frames, K, dist if world > 1 else None)
    t = torch.tensor([k_ms, e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    k_ms, e_ms = float(t[0].item()), float(t[1].item())
    if rank != 0:
        return None
    mp = n_frames * h * w / 1e6
    ok = bool(allc is not None and (allc[:, :, 0].sum(axis=1) == h * w).all())      # every frame's labels partition it
    return {"workload": "configs[3]: %d frames 1920x1080 (%d distinct synthetic frames repeated), 8 colours, one centre set, contiguous "
                        "frame shards over %d rank(s), no collective" % (n_frames, distinct, world),
            "scaling": "strong", "frames": n_frames, "frames_per_rank": -(-n_frames // world),
            "kernel": {"value": mp / (k_ms / 1e3), "unit": UNIT, "ms_total": k_ms,
                       "frac_of_hbm_peak": n_frames * h * w * (3 + 2 * K) / (k_ms / 1e3) / 1e9 / peak / world,
                       "what": "omni_color_edge_batch, 4 frames per call, frames resident in HBM, u8 planes out (max over ranks)"},
            "e2e": {"value": mp / (e_ms / 1e3), "unit": UNIT, "ms_total": e_ms,
                    "h2d_bytes": int(n_frames * h * w * 3), "d2h_bytes": int(2 * n_frames * K * h * rb),
                    "host_gbs_per_rank": (n_mine * h * w * 3 + 2 * n_mine * K * h * rb) / (e_ms / 1e3) / 1e9,
                    "what": "omni_host_color_edge_packed on each rank's shard: pinned frames in, packed masks + edges + counts out (max over ranks)"},
            "counts_gathered_in_frame_order": ok}


def stage_wall_record():
    """What a user of pipeline.py sees: the three stage scripts as subprocesses (interpreter start, CUDA context, PNG decode /
    encode included), ours (omnirevolve-image-processor_b200/image_processor/) beside the reference's as-shipped structure
    replayed on the CPU (oracle/refstages.py), on the same input and config."""
    import subprocess
    import tempfile
    import cv2
    from omni_b200.synth import synth
    out = {}
    for tag, (hh, ww_, K) in {"1024x1024 K=4 (configs[0])": (1024, 1024, 4), "4096x4096 K=8 (configs[1])": (4096, 4096, 8)}.items():
        with tempfile.TemporaryDirectory() as td:
            src = os.path.join(td, "input.png")
            cv2.imwrite(src, synth(hh, ww_, 0, 32))
            names = ["layer_dark", "layer_mid", "layer_skin", "layer_light"] if K == 4 else [f"layer_{i:02d}" for i in range(K)]
            rng = np.random.default_rng(7)
            cfg = {"input_image": src, "max_dimension": max(hh, ww_), "color_names": names,
                   "colors": [[int(v) for v in rng.integers(0, 256, 3)] for _ in range(K)]}
            rec = {}
            for arm, scripts in (("ours", [os.path.join(ROOT, "omnirevolve-image-processor_b200", "image_processor", s)
                                           for s in ("01_resize.py", "02_color_extract.py", "03_edge_detect.py")]),
                                 ("reference_port", [[os.path.join(ROOT, "oracle", "refstages.py"), s] for s in ("01", "02", "03")])):
                od = os.path.join(td, arm)
                os.makedirs(od)
                c = dict(cfg, output_dir=od)
                cp = os.path.join(od, "config.json")
                json.dump(c, open(cp, "w"))
                env = dict(os.environ, CONFIG_PATH=cp, PYTHONUNBUFFERED="1")
                ts = []
                for sc in scripts:
                    cmd = [sys.executable] + (sc if isinstance(sc, list) else [sc])
                    t0 = time.perf_counter()
                    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                    ts.append(time.perf_counter() - t0)
                    if r.returncode != 0:
                        ts[-1] = None
                        break
                rec[arm] = {"stage_s": ts, "total_s": (sum(ts) if None not in ts else None)}
            # the same three stages in ONE process (front_half.py: in-memory hand-off, one interpreter start, one CUDA context)
            od = os.path.join(td, "ours_one_process")
            os.makedirs(od)
            cp = os.path.join(od, "config.json")
            json.dump(dict(cfg, output_dir=od), open(cp, "w"))
            t0 = time.perf_counter()
            r = subprocess.run([sys.executable, os.path.join(ROOT, "omnirevolve-image-processor_b200", "image_processor", "front_half.py")],
                               env=dict(os.environ, CONFIG_PATH=cp, PYTHONUNBUFFERED="1"), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            rec["ours_one_process"] = {"total_s": (time.perf_counter() - t0) if r.returncode == 0 else None}
            if hh * ww_ <= 1024 * 1024:
                # stage 04 on these edge planes (SURVEY 8f rank 1: 152 s in the reference at this size): GPU thinning + the tracing
                # mirror with GPU degree maps, layer by layer as vectorize_all does (04:207-232), log lines discarded
                import contextlib
                import io
                from omni_b200 import contours
                t0 = time.perf_counter()
                n_paths = 0
                with contextlib.redirect_stdout(io.StringIO()):
                    for n in names:
                        e = cv2.imread(os.path.join(td, "ours", n, "edges.png"), cv2.IMREAD_GRAYSCALE)
                        sk = contours.thinning_zhangsuen(e, layer=n)
                        n_paths += len([p_ for p_ in contours.trace_centerlines(sk, layer=n) if len(p_) >= 5])
                rec["stage04_ours_s"] = time.perf_counter() - t0
                rec["stage04_polylines"] = n_paths
            same = None
            try:
                same = all(np.array_equal(cv2.imread(os.path.join(td, "ours", n, f), 0), cv2.imread(os.path.join(td, "reference_port", n, f), 0))
                           for n in names for f in ("mask.png", "edges.png"))
            except Exception:
                pass
            rec["identical_masks_and_edges"] = same
            rec["MP/s"] = {a: (hh * ww_ / 1e6 / rec[a]["total_s"]) if rec[a]["total_s"] else None for a in ("ours", "ours_one_process", "reference_port")}
            out[tag] = rec
    out["what"] = ("stages 01-03 as one subprocess each with CONFIG_PATH (pipeline.py:88-111): interpreter + imports + CUDA context "
                   "+ PNG decode/encode included; reference_port = oracle/refstages.py (the reference's stage structure replayed "
                   "with its cv2/NumPy arithmetic; the reference tree is not on this box)")
    return out


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    import omni_b200
    from omni_b200.synth import synth
    from omni_b200 import stages

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = omni_b200.Engine(local)
    peak, peak_src = peaks()
    h, w, K = wl["h"], wl["w"], wl["K"]
    B = int(wl.get("batch", 1))                                # frames per step per GPU (1: a single image)
    N = h * w * B
    img = synth(h, w, wl["seed"] + rank, wl["cell"])          # every rank its own frame(s) (sharded by frame)
    centers = stages.kmeans_lab_centers(img, K)               # host k-means, an input of the path
    _order, lut = stages.darkness_lut(centers)
    lut = lut.astype(np.uint8)
    frames = img if B == 1 else np.stack([img] + [synth(h, w, wl["seed"] + rank + 1000 * b, wl["cell"]) for b in range(1, B)])
    flush = torch.empty(384 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    sampler = ClockSampler(physical_gpu_index(local))
    sampler.start()
    time.sleep(0.05)
    m = measure_fused(torch, eng, wl, frames, centers, lut, args.steps, args.warmup, flush, barrier, cache_tables=(B > 1),
                      dump=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.result()
    if m["last"] is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in output_sample(torch, m.pop("last")).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    t = torch.tensor([m["total_ms"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = world * N / 1e6 / (ms_per_step / 1e3)
    ec = m["ec"]

    # ---- e2e: host buffers through the C ABI, H2D + kernels + D2H every step ----
    h_img = omni_b200.pinned_empty((B, h, w, 3))
    h_img[:] = frames if B > 1 else frames[None]
    rb = (w + 7) // 8
    h_mb = omni_b200.pinned_empty((B * K, h, rb))
    h_eb = omni_b200.pinned_empty((B * K, h, rb))

    def e2e_step():
        eng.host_color_edge_packed(h_img, centers, lut, ec, mask_bits=h_mb, edge_bits=h_eb, want_counts=False)

    def time_e2e(fn, steps):
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        barrier()
        s = time.perf_counter() - t0
        tt = torch.tensor([s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    e2e_s = time_e2e(e2e_step, args.steps)
    e2e_val = world * N * args.steps / 1e6 / e2e_s
    band_resends = eng.last_band_resends()
    # the same call without row bands (copy in, compute, copy out one after the other: what round 2 reported until r2_c)
    eng.set_host_bands(0)
    nb_steps = max(3, args.steps // 2)
    e2e_nb_s = time_e2e(e2e_step, nb_steps)
    eng.set_host_bands(2)
    # the u8-plane host call (what round 1 reported as e2e): 2 K bytes per pixel leave the GPU instead of 2 K bits
    h_masks = omni_b200.pinned_empty((K, h, w))
    h_edges = omni_b200.pinned_empty((K, h, w))

    def e2e_u8_step():
        for b in range(B):
            eng.host_color_edge(h_img[b], centers, lut, ec, want_labels=False, masks=h_masks, edges=h_edges, want_counts=False)

    u8_steps = max(3, args.steps // 4)
    e2e_u8_s = time_e2e(e2e_u8_step, u8_steps)
    e2e_u8_val = world * N * u8_steps / 1e6 / e2e_u8_s
    del h_masks, h_edges

    extra = {}
    if rank == 0 and world == 1:
        # ---- the other single-image configs of BASELINE.json, same measurement, fewer steps ----
        for name in ("config2", "config3"):
            if name == args.workload:
                continue
            w2 = WORKLOADS[name]
            img2 = synth(w2["h"], w2["w"], w2["seed"], w2["cell"])
            c2 = stages.kmeans_lab_centers(img2, w2["K"])
            _o2, lut2 = stages.darkness_lut(c2)
            st2 = max(5, args.steps // 2)
            m2 = measure_fused(torch, eng, w2, img2, c2, lut2.astype(np.uint8), st2, 3, flush, barrier, cache_tables=False)
            ms2 = m2["total_ms"] / st2
            N2 = w2["h"] * w2["w"]
            extra[name] = {"workload": w2["name"], "ms_per_step": ms2, "value": N2 / 1e6 / (ms2 / 1e3), "unit": UNIT,
                           "roofline": roofline_record(m2["prof"], m2["prof_step_ms"], ms2, st2, N2, w2["K"], name, peak, peak_src),
                           "step_ms": {"min": min(m2["step_ms"]), "median": statistics.median(m2["step_ms"]), "max": max(m2["step_ms"])}}
            del m2, img2
            torch.cuda.empty_cache()

    # ---- stage 01 on its own (not part of the step: the named config needs no resize) ----
    resize_extra = None
    if rank == 0 and world == 1:
        resize_extra = {}
        for tag, (sh, sw, dh, dw) in {"2:1 exact 8192x8192->4096x4096": (8192, 8192, 4096, 4096),
                                      "fractional 4096x4096->2000x2000 (default max_dimension)": (4096, 4096, 2000, 2000)}.items():
            src = torch.randint(0, 256, (sh, sw, 3), dtype=torch.uint8, device="cuda")
            dst = torch.empty((dh, dw, 3), dtype=torch.uint8, device="cuda")
            for _ in range(3):
                eng.resize_area(src, dw, dh, out=dst)
            tms = []
            for _ in range(5):
                flush.fill_(2)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); eng.resize_area(src, dw, dh, out=dst); b.record()
                torch.cuda.synchronize()
                tms.append(a.elapsed_time(b))
            ms = statistics.median(tms)
            nbytes = 3 * (sh * sw + dh * dw)
            resize_extra[tag] = {"ms": ms, "GB/s": nbytes / ms / 1e6, "frac_of_peak": nbytes / ms / 1e6 / peak,
                                 "MP/s_src": sh * sw / ms / 1e3}
            del src, dst

    # ---- process_colors.py:69-77 assign_labels (RGB palette, int16 wrap) on its own: 4096 x 4096, 16 colours ----
    i16_extra = None
    if rank == 0 and world == 1:
        pal = np.random.default_rng(1234).integers(0, 256, (16, 3)).astype(np.uint8)       # SURVEY 8d: the fixed palette of config 2
        src = torch.from_numpy(synth(4096, 4096, 0, 32)[:, :, ::-1].copy()).cuda()
        lab = torch.empty((4096, 4096), dtype=torch.uint8, device="cuda")
        for _ in range(3):
            eng.assign_rgb_i16wrap(src, pal, out=lab)
        tms = []
        for _ in range(5):
            flush.fill_(4)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); eng.assign_rgb_i16wrap(src, pal, out=lab); b.record()
            torch.cuda.synchronize()
            tms.append(a.elapsed_time(b))
        ms = statistics.median(tms)
        nb = 4096 * 4096 * 4
        i16_extra = {"ms": ms, "GB/s": nb / ms / 1e6, "frac_of_peak": nb / ms / 1e6 / peak, "MP/s": 4096 * 4096 / ms / 1e3,
                     "what": "omni_assign_rgb_i16wrap, 4096x4096 RGB, 16 palette colours -> u8 labels (3 + 1 bytes per pixel)"}
        del src, lab

    # ---- stage 04 thinning of the K edge planes the step just produced (SURVEY 8f rank 1; not part of the step) ----
    thin_extra = None
    if rank == 0 and world == 1:
        d_planes = m["d_edges"].reshape(-1, h, w)                 # [B*K, H, W]: every layer of every frame is a plane
        d_skel = torch.empty_like(d_planes)
        _o, removed, iters = eng.thin_zhangsuen(d_planes, out=d_skel, with_log=True)
        tms = []
        for _ in range(5):
            flush.fill_(3)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); eng.thin_zhangsuen(d_planes, out=d_skel); b.record()
            torch.cuda.synchronize()
            tms.append(a.elapsed_time(b))
        ms = statistics.median(tms)
        # the same from / to packed planes (1 bit per pixel): the device-side stage 03 -> 04 hand-off without byte planes
        packed_ms = None
        if B == 1:
            _mbits, ebits = eng.color_edge_packed(torch.from_numpy(frames).cuda()[None], centers, lut, ec)
            sk_bits = torch.empty_like(ebits)
            eng.thin_zhangsuen_packed(ebits, w, out=sk_bits)
            tp = []
            for _ in range(5):
                flush.fill_(3)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); eng.thin_zhangsuen_packed(ebits, w, out=sk_bits); b.record()
                torch.cuda.synchronize()
                tp.append(a.elapsed_time(b))
            packed_ms = statistics.median(tp)
            del _mbits, ebits, sk_bits
        thin_extra = {"ms": ms, "packed_ms": packed_ms, "iterations_max": int(iters.max()), "removed_px": int(removed.sum()),
                      "algorithmic_bytes": 2 * K * N, "GB/s": 2 * K * N / ms / 1e6, "frac_of_peak": 2 * K * N / ms / 1e6 / peak,
                      "layer_MP/s": K * N / ms / 1e3,
                      "what": "omni_thin_zhangsuen on the K edge planes (bytes in -> bit-planes -> cooperative Zhang-Suen -> bytes out)"}
        del d_skel
    del m["d_edges"]
    torch.cuda.empty_cache()

    # ---- BASELINE configs[3]: the 512-frame batch, sharded over the ranks (every N, strong scaling) ----
    c3 = configs3_record(torch, dist, eng, rank, world, flush, barrier, args.frames, peak)

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": wl["name"], "h": h, "w": w, "K": K, "low": wl["low"], "high": wl["high"], "ksize": wl["ksize"],
                       "frames_per_step_per_gpu": B,
                       "sharding": "one image per rank (replicas: a single image does not shard, SURVEY 8e); the sharded batch is `configs3`",
                       "l2": "flushed between steps (384 MB write, untimed); working set %d MB per step" % (N * (3 + 2 * K) // 1000000),
                       "tables": "candidate-centre tables rebuilt every step (new centres per image)" if B == 1 else "cached (one centre set)",
                       "hysteresis_passes": m["passes"], "fast_path": True},
            "gpu_launches": m["launches"], "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h_img.nbytes),
                    "d2h_bytes_per_step": int(h_mb.nbytes + h_eb.nbytes), "ms_per_step": e2e_s / args.steps * 1e3,
                    "api": "omni_host_color_edge_packed (pinned host image in; K masks + K edge planes out to pinned host memory as 1 bit per "
                           "pixel, the row format of the 1-bit PNGs the drop-in stage scripts write)",
                    "row_bands": ("one image per call: upload of band b+1 | kernels of band b | download of band b-1 overlap; edge rows leave with "
                                  "their band, bands changed by a later band are sent again (%d of the last call)" % band_resends)
                                 if band_resends >= 0 else "not used (frame groups are pipelined instead)",
                    "ms_per_step_without_bands": e2e_nb_s / nb_steps * 1e3},
            "e2e_u8": {"value": e2e_u8_val, "unit": UNIT, "h2d_bytes_per_step": int(h_img.nbytes), "d2h_bytes_per_step": int(2 * B * K * h * w),
                       "ms_per_step": e2e_u8_s / u8_steps * 1e3, "api": "omni_host_color_edge (u8 planes out)"},
            "roofline": roofline_record(m["prof"], m["prof_step_ms"], ms_per_step, args.steps, N, K, args.workload, peak, peak_src),
            "step_ms": {"min": min(m["step_ms"]), "median": statistics.median(m["step_ms"]), "max": max(m["step_ms"])},
            "wall_s_timed_region": m["wall"],
            "configs1": extra.get("config2"), "configs2": extra.get("config3"), "configs3": c3,
            "resize_kernel": resize_extra,
            "thinning_kernel": thin_extra,
            "assign_i16wrap_kernel": i16_extra,
        }
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_leg(wl, img, centers)
            out["stage_wall"] = stage_wall_record()
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="config5")
    ap.add_argument("--frames", type=int, default=512, help="frames of the configs[3] batch record")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the masks and edges of the last timed step (rank 0) to DIR/<name>.npy as float32, "
                         "a fixed seeded sample of them when they exceed 64 MB, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    wl = WORKLOADS[args.workload]
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # launched directly with --gpus N: re-launch one rank per GPU the way the driver does
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
