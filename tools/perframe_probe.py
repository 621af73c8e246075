"""Per-frame colour centres on the configs[3] frames (1920x1080, K = 8, synth seeds 0..n-1): what giving every frame its own centres
costs against one shared centre set.  Prints one JSON record (--out FILE also writes it).

  kmeans   omni_kmeans_lab_batch on 64 and on n frames (the reference's 200k subsample, 3 attempts, 40 iterations) against as many
           sequential omni_kmeans_lab calls (host clock: both synchronise), with the per-frame results compared bit for bit.
  kernel   one 4-frame group on the device: omni_color_edge_packed_frames (each frame's own centres and LUT) against the
           shared-centre omni_color_edge_packed (table cache on: its tables are built once; and off), CUDA events over `--steps`
           calls each, alternating; plus the per-kernel profile of one call of each.
  e2e      n pinned host frames -> omni_host_color_edge_packed_frames against omni_host_color_edge_packed (host clock), alternating.

    python tools/perframe_probe.py [--frames 512] [--steps 50] [--rounds 3] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(R, "omnirevolve-image-processor_b200")
sys.path.insert(0, R)
sys.path.insert(0, PKG)


def card_line(torch):
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:              # the record still names the card through torch
        q = f"nvidia-smi unavailable: {e}"
    return torch.cuda.get_device_name(0), q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    import omni_b200
    from omni_b200 import stages
    from omni_b200.synth import synth
    card, smi = card_line(torch)
    h, w, K, n = 1080, 1920, 8, a.frames
    eng = omni_b200.Engine(0)
    frames = omni_b200.pinned_empty((n, h, w, 3))
    for i in range(n):
        frames[i] = synth(h, w, i, 32)
    d_frames = torch.from_numpy(frames).cuda()
    pick = stages._sample_pick(h * w, 200_000)
    rec = {"probe": "perframe_probe", "workload": f"configs[3] frames: {n} x 1920x1080 synth(seed 0..{n - 1}), K=8, 50/150, blur 3, "
           "morph 3/1/1", "card": card, "nvidia_smi": smi, "steps": a.steps, "rounds": a.rounds}

    # ---- k-means ----
    def wall(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    eng.kmeans_lab_batch(d_frames[:2], K, pick)                                   # warm-up (module load, workspace)
    eng.kmeans_lab(d_frames[0], K, pick)
    km = {}
    centers = None
    for nb in sorted({min(64, n), n}):
        tb, seq = [], []
        for r in range(a.rounds if nb <= 64 else 1):
            t, (cb, pb) = wall(lambda: eng.kmeans_lab_batch(d_frames[:nb], K, pick))
            tb.append(t)
            t, outs = wall(lambda: [eng.kmeans_lab(d_frames[f], K, pick) for f in range(nb)])
            seq.append(t)
        cs = np.stack([c for c, _ in outs])
        ps = np.array([p for _, p in outs])
        km[str(nb)] = {"batch_s_median": round(statistics.median(tb), 4), "sequential_s_median": round(statistics.median(seq), 4),
                       "batch_s": [round(x, 4) for x in tb], "sequential_s": [round(x, 4) for x in seq],
                       "speedup": round(statistics.median(seq) / statistics.median(tb), 2),
                       "batch_ms_per_frame": round(1e3 * statistics.median(tb) / nb, 3),
                       "sequential_ms_per_frame": round(1e3 * statistics.median(seq) / nb, 3),
                       "bit_identical": bool(np.array_equal(cb.view(np.uint32), cs.view(np.uint32)) and np.array_equal(pb, ps))}
        if nb == n:
            centers = cb
    rec["kmeans"] = km
    luts = np.stack([stages.darkness_lut(c)[1] for c in centers]).astype(np.uint8)
    shared_c, shared_l = centers[0], luts[0]

    # ---- kernel time per 4-frame group ----
    ec = omni_b200.EdgeConfig()
    G = 32 // K
    grp = d_frames[:G]
    rb = (w + 7) // 8

    def per_frame():
        return eng.color_edge_packed(grp, centers[:G], luts[:G], ec)

    def shared():
        return eng.color_edge_packed(grp, shared_c, shared_l, ec)

    variants = {"per_frame": (per_frame, True), "shared_cache_on": (shared, True), "shared_cache_off": (shared, False)}
    times = {k: [] for k in variants}
    for _ in range(a.rounds):
        for key, (fn, cache) in variants.items():
            eng.set_table_cache(cache)
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            for _ in range(a.steps):
                fn()
            ev[1].record()
            torch.cuda.synchronize()
            times[key].append(ev[0].elapsed_time(ev[1]) / a.steps)
    eng.set_table_cache(True)
    kern = {k: {"ms_per_group_median": round(statistics.median(v), 4), "ms_per_group": [round(x, 4) for x in v]} for k, v in times.items()}
    kern["ratio_per_frame_over_shared_cache_on"] = round(kern["per_frame"]["ms_per_group_median"] / kern["shared_cache_on"]["ms_per_group_median"], 3)
    kern["ratio_per_frame_over_shared_cache_off"] = round(kern["per_frame"]["ms_per_group_median"] / kern["shared_cache_off"]["ms_per_group_median"], 3)
    prof = {}
    for key, (fn, cache) in variants.items():
        eng.set_table_cache(cache)
        fn()
        eng.profile(True)
        fn()
        prof[key] = eng.profile_summary()
        eng.profile(False)
    eng.set_table_cache(True)
    kern["profile_one_call"] = prof
    rec["kernel_4_frame_group"] = kern

    # ---- end to end, host buffers ----
    mb = omni_b200.pinned_empty((n * K, h, rb))
    eb = omni_b200.pinned_empty((n * K, h, rb))
    e2e = {"per_frame": [], "shared": []}
    eng.host_color_edge_packed(frames[:2 * G], centers[:2 * G], luts[:2 * G], ec, mask_bits=mb[:2 * G * K], edge_bits=eb[:2 * G * K])
    eng.host_color_edge_packed(frames[:2 * G], shared_c, shared_l, ec, mask_bits=mb[:2 * G * K], edge_bits=eb[:2 * G * K])
    counts = {}
    for _ in range(a.rounds):
        t, r = wall(lambda: eng.host_color_edge_packed(frames, centers, luts, ec, mask_bits=mb, edge_bits=eb))
        e2e["per_frame"].append(t)
        counts["per_frame"] = r["counts"]
        t, r = wall(lambda: eng.host_color_edge_packed(frames, shared_c, shared_l, ec, mask_bits=mb, edge_bits=eb))
        e2e["shared"].append(t)
        counts["shared"] = r["counts"]
    rec["e2e_host"] = {k: {"s_median": round(statistics.median(v), 4), "s": [round(x, 4) for x in v],
                           "frames_per_s": round(n / statistics.median(v), 1)} for k, v in e2e.items()}
    rec["e2e_host"]["ratio_per_frame_over_shared"] = round(rec["e2e_host"]["per_frame"]["s_median"] / rec["e2e_host"]["shared"]["s_median"], 3)
    rec["e2e_host"]["labels_partition_every_frame"] = bool(all((c[:, 0].reshape(n, K).sum(1) == h * w).all() for c in counts.values()))
    s = json.dumps(rec)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(rec, indent=1) + "\n")
    eng.close()


if __name__ == "__main__":
    main()
