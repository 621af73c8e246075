"""PNG encode on the GPU against the host encoders the stages used before (profiles/r7_png_probe.json).

    python tools/png_probe.py [--out record.json] [--reps 6]

One command records:
  1. device encode time of omni_png_encode (kernel time from the ctx's CUDA events, and the whole call: kernels, the size
     read-back and the copy of the files to the host) for 32 planes of 4096^2 at 1 bit (K=16 masks + edges), one 4096^2 BGR image
     and the mask + edge planes of one 4-frame group of configs[3] (4 x 1080p, K=8);
  2. host encode time on this machine's host for the same files: png1.encode_png1 (one thread per plane, as the stages ran it)
     and cv2.imencode with the parameters the stages used (default for resized.png, PNG_COMPRESSION 1 for the composite);
  3. the file sizes of both;
  4. stage wall time at 4096^2, K=8: the three stage scripts and front_half.py, with the old encoders swapped back in and with
     the GPU encoder, alternated, each arm `--reps` times;
plus the card name and power limit from a read-only nvidia-smi query."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "omnirevolve-image-processor_b200")
SCRIPTS = os.path.join(PKG, "image_processor")
sys.path.insert(0, PKG)

# Run a stage script with the encoders of before swapped back in (the stages' encoder hooks, and front_half_main as it was).
OLD_ENCODERS = r'''
import os, sys, threading, runpy
from concurrent.futures import ThreadPoolExecutor
sys.path[:0] = [os.path.dirname(SCRIPT), os.path.dirname(os.path.dirname(SCRIPT))]
import cv2
from omni_b200 import stages, png1
def _layers(bits, w):
    with ThreadPoolExecutor(max(1, min(len(bits), os.cpu_count() or 1))) as ex:     # as the I/O pool encoded them
        return list(ex.map(lambda b: png1.encode_png1(b, w), bits))
stages._encode_layers = _layers
stages._encode_resized = lambda img: cv2.imencode(".png", img)[1].tobytes()
stages._encode_composite = lambda c: cv2.imencode(".png", c, [cv2.IMWRITE_PNG_COMPRESSION, 1])[1].tobytes()
def _front_half_main(cfg):
    cfg.ensure_output_dirs()
    img = stages.resize_if_needed(cfg.input_image, cfg)
    path = os.path.join(cfg.output_dir, "resized.png")
    writer = threading.Thread(target=cv2.imwrite, args=(path, img))
    writer.start()
    try:
        stages.color_extract_main(cfg, img=img)
    finally:
        writer.join()
    print(f"Saved: {path}")
    stages.edge_detect_main(cfg)
stages.front_half_main = _front_half_main
runpy.run_path(SCRIPT, run_name="__main__")
'''
NEW_ENCODERS = r'''
import os, sys, runpy
sys.path.insert(0, os.path.dirname(SCRIPT))
runpy.run_path(SCRIPT, run_name="__main__")
'''


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else f"nvidia-smi failed: {r.stdout.strip()}"


def time_device(eng, t, fmt, w, reps):
    import torch
    for _ in range(3):
        files = eng.png_encode(t, fmt, w)
    torch.cuda.synchronize()
    eng.profile(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(reps):
        eng.png_encode(t, fmt, w)
    ev1.record()
    torch.cuda.synchronize()
    call_ms = (time.perf_counter() - t0) * 1e3 / reps
    prof = eng.profile_summary()
    eng.profile(False)
    kern = {k: v[1] / reps for k, v in prof.items() if k.startswith("png_")}
    return files, {"kernel_ms": sum(kern.values()), "kernels_ms": kern, "events_ms_per_call": ev0.elapsed_time(ev1) / reps,
                   "call_ms_host_clock": call_ms}


def time_host(fn, items, threads, reps=2):
    best, out = None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        if threads > 1:
            with ThreadPoolExecutor(threads) as ex:
                out = list(ex.map(fn, items))
        else:
            out = [fn(x) for x in items]
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return out, best * 1e3


def workloads(eng):
    import cv2
    from omni_b200 import stages, synth as osynth
    ec = __import__("omni_b200").EdgeConfig()
    img = osynth.synth(4096, 4096, 0)
    c16 = stages.kmeans_lab_centers(img, 16)
    _o, lut16 = stages.darkness_lut(c16)
    r16 = eng.host_color_edge_packed(img, c16, lut16.astype(np.uint8), ec, msb_first=True)
    c8 = stages.kmeans_lab_centers(img, 8)
    _o, lut8 = stages.darkness_lut(c8)
    r8 = eng.host_color_edge_packed(img, c8, lut8.astype(np.uint8), ec, msb_first=True)
    rng = np.random.default_rng(7)
    stack = np.unpackbits(r8["edge_bits"], axis=2)[:, :, :4096] * np.uint8(255)
    canvas = eng.host_edges_composite(stack, [tuple(int(v) for v in rng.integers(0, 256, 3)) for _ in range(8)])
    frames = np.stack([osynth.synth(1080, 1920, s) for s in range(4)])
    cf = stages.kmeans_lab_centers(frames[0], 8)
    _o, lutf = stages.darkness_lut(cf)
    rf = eng.host_color_edge_packed(frames, cf, lutf.astype(np.uint8), ec, msb_first=True)
    return {
        "4096x4096 1-bit, 32 planes (K=16 masks + edges)": ("gray1", np.concatenate([r16["mask_bits"], r16["edge_bits"]]), 4096),
        "4096x4096 BGR (resized.png)": ("bgr8", img, None),
        "4096x4096 BGR (edges_composite.png, K=8)": ("bgr8", canvas, None),
        "1920x1080 1-bit, 64 planes (configs[3]: 4 frames, K=8, masks + edges)":
            ("gray1", np.concatenate([rf["mask_bits"], rf["edge_bits"]]), 1920),
    }, cv2


def encode_records(eng, reps):
    import torch
    from omni_b200 import png1
    loads, cv2 = workloads(eng)
    out = {}
    threads = os.cpu_count() or 1
    for name, (fmt, a, w) in loads.items():
        rec = {}
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        files, rec["gpu_device_form"] = time_device(eng, t, fmt, w, reps)
        t0 = time.perf_counter()
        hfiles = eng.host_png_encode(a, fmt, w)
        rec["gpu_host_form_ms"] = (time.perf_counter() - t0) * 1e3
        assert hfiles == files
        rec["gpu_bytes"] = int(sum(map(len, files)))
        if fmt == "gray1":
            _f, rec["png1_encode_ms_1thread"] = time_host(lambda b: png1.encode_png1(b, w), list(a), 1, 1)
            old, rec[f"png1_encode_ms_{threads}threads"] = time_host(lambda b: png1.encode_png1(b, w), list(a), threads)
            rec["png1_bytes"] = int(sum(map(len, old)))
            rec["size_ratio_gpu_over_png1"] = rec["gpu_bytes"] / rec["png1_bytes"]
            ok = all(np.array_equal(cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_UNCHANGED),
                                    np.unpackbits(p, axis=1)[:, :w] * np.uint8(255)) for f, p in zip(files, a))
        else:
            params = [] if "resized" in name else [cv2.IMWRITE_PNG_COMPRESSION, 1]
            old, rec["cv2_imencode_stage_params_ms"] = time_host(lambda x: cv2.imencode(".png", x, params)[1], [a], 1)
            rec["cv2_stage_params"] = "default" if not params else "PNG_COMPRESSION 1"
            rec["cv2_stage_params_bytes"] = int(len(old[0]))
            dflt, rec["cv2_imencode_default_ms"] = time_host(lambda x: cv2.imencode(".png", x)[1], [a], 1, 1)
            rec["cv2_default_bytes"] = int(len(dflt[0]))
            rec["size_ratio_gpu_over_cv2_default"] = rec["gpu_bytes"] / rec["cv2_default_bytes"]
            ok = np.array_equal(cv2.imdecode(np.frombuffer(files[0], np.uint8), cv2.IMREAD_UNCHANGED), a)
        rec["gpu_files_decode_to_source"] = bool(ok)
        out[name] = rec
    return out


def stage_wall(reps):
    import cv2
    from omni_b200.synth import synth
    res = {a: {"three_scripts_s": [], "per_script_s": [], "front_half_s": []} for a in ("old", "new")}
    same = True
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "input.png")
        cv2.imwrite(src, synth(4096, 4096, 0, 32))
        names = [f"layer_{i:02d}" for i in range(8)]
        rng = np.random.default_rng(7)
        cfg = {"input_image": src, "max_dimension": 4096, "color_names": names,
               "colors": [[int(v) for v in rng.integers(0, 256, 3)] for _ in range(8)]}

        def run(arm, script, od):
            code = (OLD_ENCODERS if arm == "old" else NEW_ENCODERS).replace("SCRIPT", repr(os.path.join(SCRIPTS, script)))
            env = dict(os.environ, CONFIG_PATH=os.path.join(od, "config.json"), PYTHONUNBUFFERED="1", OMNI_B200_HOME=PKG)
            t0 = time.perf_counter()
            r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"{arm} {script} failed:\n{r.stdout[-3000:]}")
            return time.perf_counter() - t0

        dirs = {}
        for rep in range(reps):
            for arm in (("old", "new") if rep % 2 == 0 else ("new", "old")):
                for kind in ("three", "front"):
                    od = os.path.join(td, f"{arm}_{kind}_{rep}")
                    os.makedirs(od)
                    json.dump(dict(cfg, output_dir=od), open(os.path.join(od, "config.json"), "w"))
                    if kind == "three":
                        per = [run(arm, s, od) for s in ("01_resize.py", "02_color_extract.py", "03_edge_detect.py")]
                        res[arm]["per_script_s"].append(per)
                        res[arm]["three_scripts_s"].append(sum(per))
                    else:
                        res[arm]["front_half_s"].append(run(arm, "front_half.py", od))
                    dirs[(arm, kind)] = od
        for kind in ("three", "front"):
            a, b = dirs[("old", kind)], dirs[("new", kind)]
            files = ["resized.png", "edges_composite.png"] + [os.path.join(n, f) for n in names for f in ("mask.png", "edges.png")]
            for f in files:
                x = cv2.imread(os.path.join(a, f), cv2.IMREAD_UNCHANGED)
                y = cv2.imread(os.path.join(b, f), cv2.IMREAD_UNCHANGED)
                same = same and x is not None and y is not None and np.array_equal(x, y)
    for arm in res:
        for k in ("three_scripts_s", "front_half_s"):
            res[arm][k[:-2] + "_median_s"] = float(np.median(res[arm][k]))
        res[arm]["per_script_median_s"] = [float(v) for v in np.median(np.array(res[arm]["per_script_s"]), axis=0)]
    res["decoded_pixels_identical_old_vs_new"] = bool(same)
    res["what"] = ("4096x4096 synth input, K=8, max_dimension 4096: wall time of each stage script as a subprocess (interpreter, "
                   "CUDA context, PNG decode / encode included), summed over 01-03, and of front_half.py; arms alternated")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the record (default: print it only)")
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--enc-reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("png_probe needs a CUDA device")
    from omni_b200 import get_engine
    rec = {"gpu": gpu_info(), "host_cpus": os.cpu_count(),
           "encode": encode_records(get_engine(0), args.enc_reps), "stage_wall_4096_k8": stage_wall(args.reps)}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
