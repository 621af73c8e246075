"""Centrelines of a whole frame batch from its packed edge planes (omni_centerlines_packed) against the per-frame loop of the
existing calls, on the card this runs on.  Prints one JSON record (--out FILE also writes it).

Frames: configs[3]-style 1920x1080 synthetic frames (synth seeds 0..n-1, cell 32), K = 8, one centre set (cv2.kmeans centres of
frame 0, darkness order), edge planes from omni_host_color_edge_packed (MSB first), at n = 64 and n = 512 frames.
Arms, alternated over `--rounds` repeats; host clock around C calls that end in a stream synchronisation, up to the point where
the polylines are in the ctx (copying them out is not timed: these frames give ~10^7 points per frame, so it is a copy of
~75 MB per frame that both arms would pay alike):
  batch_device   omni_centerlines_packed on the n*K planes resident on the device
  batch_host     omni_host_centerlines_packed on the n*K planes in pinned host memory
  loop_device    per frame: omni_thin_zhangsuen_packed of its K planes -> bits unpacked to {0,255} bytes on the device (a torch
                 expression of the probe; the library has no unpack call) -> omni_trace_centerlines
  loop_host      (n <= 64 only) per frame: np.unpackbits on the host -> omni_host_thin_zhangsuen -> omni_host_trace_centerlines
Equality, in the same run, of batch_device against loop_device frame by frame: the per-plane rows (total_fg, components,
polylines, points), the polyline lengths and the component rows of every plane, and at n <= 64 the points themselves; and the
per-plane rows of batch_host against batch_device.  Then one profiled batch_device call: per-kernel CUDA-event times
(omni_profile_summary) grouped into thinning, unpacking, labelling and walks.  The card name, power limit and SM clock limit are
read in the same run.

    python tools/centerlines_probe.py [--frames 64,512] [--rounds 3] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "omnirevolve-image-processor_b200")]

import numpy as np  # noqa: E402

H, W, K = 1080, 1920, 8
RB = (W + 7) // 8


def card_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi failed: " + q.stdout.strip()
    except Exception as e:
        return f"nvidia-smi unavailable: {e}"


GROUPS = {"thinning": ("unpack_planes", "thin_zhangsuen", "pack_planes"), "unpacking": ("trace_bits_to_bytes",),
          "labelling": ("trace_ccl_init", "trace_ccl_merge", "trace_ccl_flatten", "trace_label_count", "trace_label_scan",
                        "trace_label_assign", "trace_comp_init", "trace_comp_stats"),
          "walks": ("trace_row_count", "trace_row_scan", "trace_row_fill", "trace_walk_count", "trace_walk_count_global",
                    "trace_walk_write", "trace_walk_write_global")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", default="64,512")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import omni_b200
    from omni_b200 import capi, stages
    from omni_b200.synth import synth
    assert torch.cuda.is_available(), "centerlines_probe needs a CUDA device"
    sizes = [int(x) for x in a.frames.split(",")]
    n_max = max(sizes)
    rec = {"probe": "centerlines_probe", "card": card_line(), "torch_device": torch.cuda.get_device_name(0), "rounds": a.rounds,
           "workload": f"configs[3]-style frames: 1920x1080 synth(seed 0..n-1, cell 32), K=8, one centre set (cv2.kmeans of frame 0), "
                       "Canny 50/150, blur 3, morph 3/1/1; packed MSB-first edge planes from omni_host_color_edge_packed; max_iter 120"}
    eng = omni_b200.Engine(0)
    L, hctx = capi.lib(), eng._h
    i64 = C.POINTER(C.c_int64)
    frames = omni_b200.pinned_empty((n_max, H, W, 3))
    for i in range(n_max):
        frames[i] = synth(H, W, i, 32)
    centers = stages.kmeans_lab_centers(frames[0], K)
    _o, lut = stages.darkness_lut(centers)
    bits = omni_b200.pinned_empty((n_max * K, H, RB))
    eng.host_color_edge_packed(frames, centers, lut.astype(np.uint8), omni_b200.EdgeConfig(), edge_bits=bits, want_counts=False)
    del frames
    d_bits_all = torch.from_numpy(bits).cuda()
    shifts = torch.arange(7, -1, -1, dtype=torch.uint8, device="cuda")
    stream = eng._stream()

    def batch_device(d, info):
        capi.check(L.omni_centerlines_packed(hctx, d.data_ptr(), d.shape[0], H, W, H * RB, RB, 1, 120, info.ctypes.data_as(i64),
                                             stream))

    def batch_host(hb, info):
        capi.check(L.omni_host_centerlines_packed(hctx, hb.ctypes.data, hb.shape[0], H, W, H * RB, RB, 1, 120, info.ctypes.data_as(i64)))

    def loop_device_frame(d, f, info):
        thin = eng.thin_zhangsuen_packed(d[f * K:(f + 1) * K], W)
        sk = (((thin[..., None] >> shifts) & 1) * 255).reshape(K, H, RB * 8)[:, :, :W].contiguous()
        capi.check(L.omni_trace_centerlines(hctx, sk.data_ptr(), K, H, W, sk.stride(0), sk.stride(1),
                                            info[f * K:(f + 1) * K].ctypes.data_as(i64), stream))

    def loop_device(d, info):
        for f in range(d.shape[0] // K):
            loop_device_frame(d, f, info)

    def loop_host(hb, info):
        for f in range(hb.shape[0] // K):
            e = np.unpackbits(hb[f * K:(f + 1) * K], axis=2)[:, :, :W] * np.uint8(255)
            sk = eng.host_thin_zhangsuen(e)[0]
            capi.check(L.omni_host_trace_centerlines(hctx, sk.ctypes.data, K, H, W, sk.strides[0], sk.strides[1],
                                                     info[f * K:(f + 1) * K].ctypes.data_as(i64)))

    def results(info, points):
        """The result in the ctx: (points | None, polyline lengths, component rows)."""
        n_comp, n_paths, n_pts = (int(v) for v in info[:, 1:].sum(axis=0))
        pts = np.empty((n_pts, 2), np.int32) if points else None
        lens = np.empty(n_paths, np.int32)
        comp = np.empty((n_comp, 6), np.int32)
        capi.check(L.omni_trace_results(hctx, pts.ctypes.data if points else None, lens.ctypes.data, comp.ctypes.data))
        return pts, lens, comp

    def wall(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    for n in sizes:
        P = n * K
        d, hb = d_bits_all[:P], bits[:P]
        infos = {}
        arms = {"batch_device": lambda i: batch_device(d, i), "batch_host": lambda i: batch_host(hb, i),
                "loop_device": lambda i: loop_device(d, i)}
        if n <= 64:
            arms["loop_host"] = lambda i: loop_host(hb, i)
        for k, fn in arms.items():                                     # warm-up: modules, workspaces of this size
            infos[k] = np.zeros((P, 4), np.int64)
            fn(infos[k])
        times = {k: [] for k in arms}
        for _ in range(a.rounds):
            for k, fn in arms.items():
                times[k].append(wall(lambda: fn(infos[k])))
        # equality: the batch result against the loop, frame by frame (each loop call replaces the result in the ctx)
        full = n <= 64
        info_b = np.zeros((P, 4), np.int64)
        batch_device(d, info_b)
        pts_b, lens_b, comp_b = results(info_b, full)
        cum = np.zeros((n + 1, 3), np.int64)
        cum[1:] = np.cumsum(info_b[:, 1:].reshape(n, K, 3).sum(axis=1), axis=0)
        same = True
        info_f = np.zeros((P, 4), np.int64)
        for f in range(n):
            loop_device_frame(d, f, info_f)
            p, ln, cp = results(info_f[f * K:(f + 1) * K], full)
            (c0, l0, q0), (c1, l1, q1) = cum[f], cum[f + 1]
            same = same and np.array_equal(ln, lens_b[l0:l1]) and np.array_equal(cp, comp_b[c0:c1]) and \
                (not full or np.array_equal(p, pts_b[q0:q1]))
        same = same and np.array_equal(info_f, info_b)
        del pts_b
        r = {"planes": P, "chunks": -(-P // min(P, max(32, (256 << 20) // (8 * ((W + 1) // 2) * ((H + 1) // 2))))),
             "skeleton_px": int(info_b[:, 0].sum()), "components": int(info_b[:, 1].sum()), "polylines": int(info_b[:, 2].sum()),
             "points": int(info_b[:, 3].sum()),
             "batch_device_equals_loop_device": bool(same), "compared": "per-plane rows, polyline lengths, component rows" +
             (", points" if full else " (points not compared at this size)"),
             "plane_rows_equal_every_arm": bool(all(np.array_equal(v, info_b) for v in infos.values()))}
        for k, v in times.items():
            r[k] = {"s_median": round(statistics.median(v), 4), "s": [round(x, 4) for x in v],
                    "ms_per_frame": round(1e3 * statistics.median(v) / n, 3)}
        r["speedup_batch_device_over_loop_device"] = round(r["loop_device"]["s_median"] / r["batch_device"]["s_median"], 2)
        r["speedup_batch_host_over_loop_device"] = round(r["loop_device"]["s_median"] / r["batch_host"]["s_median"], 2)
        if "loop_host" in r:
            r["speedup_batch_host_over_loop_host"] = round(r["loop_host"]["s_median"] / r["batch_host"]["s_median"], 2)
        eng.profile(True)
        batch_device(d, info_b)
        prof = eng.profile_summary()
        eng.profile(False)
        split = {g: round(sum(prof.get(k, (0, 0.0))[1] for k in names), 3) for g, names in GROUPS.items()}
        split["other"] = round(sum(v[1] for k, v in prof.items() if not any(k in names for names in GROUPS.values())), 3)
        r["batch_device_kernel_ms"] = split
        r["batch_device_kernels"] = {k: [v[0], round(v[1], 4)] for k, v in prof.items()}
        rec[f"n{n}"] = r
        print(json.dumps({f"n{n}": {k: v for k, v in r.items() if k != "batch_device_kernels"}}), flush=True)
    rec["card_after"] = card_line()
    s = json.dumps(rec)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(rec, indent=1) + "\n")
    eng.close()


if __name__ == "__main__":
    main()
