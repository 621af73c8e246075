#!/usr/bin/env python3
"""Timing of stage 04 `trace_centerlines` on the GPU (omni_trace_centerlines) against the host walk, on the card this runs on.

    python tools/trace_probe.py [--out FILE.json] [--host-4096 N] [--reps N]

Inputs:
  * the four 1024^2, K=4 pipeline layers: synth(1024, 1024, 0), the reference's k-means centres and darkness order
    (oracle/refport.py), edges from omni_host_color_edge, skeletons from omni_thin_zhangsuen;
  * 4096^2 edge planes, K=8 and K=16, from omni_color_edge on synth(4096, 4096, 1, cell=64) with fixed Lab centres, thinned
    on the device.
Per set: kernel time (CUDA events around every kernel of the call, omni_profile_*), wall time of Engine.trace_centerlines
(the call, the result copy and the NumPy polylines), the output sizes.  The host walk (contours.trace_centerlines with cv2's
maps) on the 1024^2 layers and on the N smallest 4096^2 K=8 layers, checked equal to the GPU polylines.  The stage-04 shim's
wall time at 1024^2, K=4 (thinning + tracing of the four layers through image_processor/04_find_contours.py, with a stand-in
for the reference's file whose vectorize_all does only those two steps).  The card name and power limit come from the same
run.  A GPU is required."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "omnirevolve-image-processor_b200")]

import cv2  # noqa: E402
import numpy as np  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi failed: " + q.stdout.strip()


def maps(sk):
    S = (sk > 0).astype(np.uint8)
    k = np.ones((3, 3), np.uint8)
    k[1, 1] = 0
    deg = cv2.filter2D(S, cv2.CV_8U, k, borderType=cv2.BORDER_CONSTANT)
    return deg, (S == 1) & (deg == 1), (S == 1) & (deg >= 3)


def gpu_trace(eng, skel, reps):
    """skel: CUDA [K,H,W].  Returns (result, record)."""
    res = eng.trace_centerlines(skel)                       # warm-up (module load, workspace growth)
    walls = []
    for _ in range(reps):
        t = time.perf_counter()
        res = eng.trace_centerlines(skel)
        walls.append(time.perf_counter() - t)
    eng.profile(True)
    eng.trace_centerlines(skel)
    prof = eng.profile_summary()
    eng.profile(False)
    kms = {k: round(v[1], 4) for k, v in prof.items() if k.startswith("trace_")}
    return res, {
        "K": int(skel.shape[0]), "H": int(skel.shape[1]), "W": int(skel.shape[2]),
        "skeleton_px": [r.total_fg for r in res], "components": [len(r.stats) for r in res],
        "polylines": [len(r.paths) for r in res], "points": [int(sum(len(p) for p in r.paths)) for r in res],
        "kernel_ms_total": round(sum(kms.values()), 3), "kernel_ms": kms,
        "wall_ms_median": round(1e3 * float(np.median(walls)), 3), "wall_ms_min": round(1e3 * min(walls), 3), "reps": reps,
    }


def host_walk(sk, gpu_paths):
    from omni_b200 import contours
    t = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        paths = contours.trace_centerlines(sk, "L", maps=maps(sk))
    dt = time.perf_counter() - t
    same = len(paths) == len(gpu_paths) and all(np.array_equal(a, b) for a, b in zip(paths, gpu_paths))
    return {"skeleton_px": int((sk > 0).sum()), "seconds": round(dt, 3), "equal_to_gpu": bool(same)}


def shim_wall(edges):
    """Stage-04 shim (image_processor/04_find_contours.py) on K edge planes, as a separate process: seconds of vectorize_all."""
    import shutil
    src = os.path.join(ROOT, "omnirevolve-image-processor_b200", "image_processor")
    with tempfile.TemporaryDirectory() as d:
        for f in ("04_find_contours.py", "_omni_path.py"):
            shutil.copy(os.path.join(src, f), d)
        names = [f"layer_{i}" for i in range(len(edges))]
        with open(os.path.join(d, "04_find_contours_ref.py"), "w") as f:
            f.write("import os, pickle, time, cv2\n"
                    "def load_config():\n"
                    "    class C: pass\n"
                    f"    c = C(); c.output_dir = os.environ['OUT_DIR']; c.color_names = {names!r}; return c\n"
                    "def thinning_zhangsuen(img, layer): raise RuntimeError('not replaced')\n"
                    "def trace_centerlines(skel, layer): raise RuntimeError('not replaced')\n"
                    "def vectorize_layer(name, cfg):\n"
                    "    e = cv2.imread(os.path.join(cfg.output_dir, name, 'edges.png'), cv2.IMREAD_GRAYSCALE)\n"
                    "    return name, trace_centerlines(thinning_zhangsuen(e, layer=name), layer=name)\n"
                    "def vectorize_all(cfg):\n"
                    "    t = time.perf_counter(); out = dict(vectorize_layer(n, cfg) for n in cfg.color_names)\n"
                    "    pickle.dump(out, open(os.path.join(cfg.output_dir, 'contours.pkl'), 'wb'))\n"
                    "    print('VECTORIZE_ALL_S', time.perf_counter() - t)\n")
        out = os.path.join(d, "out")
        for n, e in zip(names, edges):
            os.makedirs(os.path.join(out, n))
            cv2.imwrite(os.path.join(out, n, "edges.png"), e)
        env = dict(os.environ, OUT_DIR=out, OMNI_B200_HOME=os.path.join(ROOT, "omnirevolve-image-processor_b200"))
        t = time.perf_counter()
        r = subprocess.run([sys.executable, os.path.join(d, "04_find_contours.py")], env=env, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True)
        wall = time.perf_counter() - t
        if r.returncode != 0:
            raise RuntimeError(r.stdout[-2000:])
        inner = [float(ln.split()[1]) for ln in r.stdout.splitlines() if ln.startswith("VECTORIZE_ALL_S")][0]
        return {"layers": len(edges), "vectorize_all_s": round(inner, 3), "process_wall_s": round(wall, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON record to this file (it is always printed)")
    ap.add_argument("--host-4096", type=int, default=1, help="4096^2 layers to walk on the host as well")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    import omni_b200
    from omni_b200 import EdgeConfig
    from omni_b200.synth import synth
    from oracle import refport as rp
    assert torch.cuda.is_available(), "trace_probe needs a CUDA device"
    eng = omni_b200.get_engine()
    rec = {"card": card(), "torch_device": torch.cuda.get_device_name(0)}

    img = synth(1024, 1024, 0)
    K = 4
    centers = rp.kmeans_lab_centers(img, K)
    _order, lut = rp.darkness_order(centers)
    edges = eng.host_color_edge(img, centers, lut, EdgeConfig())["edges"]
    skel = eng.thin_zhangsuen(torch.from_numpy(edges).cuda())
    res, rec["gpu_1024_k4"] = gpu_trace(eng, skel, a.reps)
    sks = skel.cpu().numpy()
    rec["host_1024_k4"] = [host_walk(sks[i], res[i].paths) for i in range(K)]
    rec["shim_1024_k4"] = shim_wall(edges)

    big = torch.from_numpy(synth(4096, 4096, 1, cell=64)).cuda()
    for K in (8, 16):
        ctr = np.array([[8 + 240 * i / (K - 1), 128 + 40 * np.sin(i), 128 + 40 * np.cos(i)] for i in range(K)], np.float32)
        _l, _m, e = eng.color_edge(big, ctr, np.arange(K, dtype=np.uint8), EdgeConfig())
        skel = eng.thin_zhangsuen(e)
        res, rec[f"gpu_4096_k{K}"] = gpu_trace(eng, skel, a.reps)
        if K == 8 and a.host_4096:
            sks = skel.cpu().numpy()
            order = sorted((i for i in range(K) if res[i].total_fg), key=lambda i: res[i].total_fg)[:a.host_4096]
            rec["host_4096_k8"] = [dict(layer=i, **host_walk(sks[i], res[i].paths)) for i in order]
        del skel, e, _m, _l
    rec["card_after"] = card()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
