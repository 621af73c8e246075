"""Stage-03 morphology sizes, parent library against the current one: omni_edges on the 4096^2, K=16 masks of the `synth` image at
edge_morph_kernel 3 (2 open + 2 close iterations) and 5, 7, 9, 15, 31, 63 (1 + 1).  Each library runs in its own worker process
(a library is picked through OMNI_B200_LIB at import); the workers alternate base, new, base, new.  Per size: median of 20
CUDA-event timings after warm-up, and a checksum of the edge planes, so that equal outputs are recorded where the parent supports
the parameters.  Prints one JSON record.

    python tools/morph_probe.py [--base LIB] [--new LIB] [--rounds N] [--out FILE]

Build the parent commit's library beforehand, e.g. from a `git worktree` of it into omnirevolve-image-processor_b200/lib/libomni_base.so."""
import argparse
import json
import os
import statistics
import subprocess
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(R, "omnirevolve-image-processor_b200")
CASES = [(3, 2, 2), (5, 1, 1), (7, 1, 1), (9, 1, 1), (15, 1, 1), (31, 1, 1), (63, 1, 1)]


def worker(steps, warmup):
    sys.path.insert(0, R); sys.path.insert(0, PKG)
    import numpy as np, torch, omni_b200          # noqa: E401
    from omni_b200.synth import synth
    from omni_b200 import stages
    h = w = 4096
    K = 16
    eng = omni_b200.Engine(0)
    img = synth(h, w, 0, 32)
    ctr = stages.kmeans_lab_centers(img, K)
    _o, lut = stages.darkness_lut(ctr)
    masks = eng.color_edge(torch.from_numpy(img).cuda(), ctr, lut.astype(np.uint8), omni_b200.EdgeConfig())[1]
    edges = torch.empty_like(masks)
    out = {}
    for mk, oi, ci in CASES:
        ec = omni_b200.EdgeConfig(ksize=3, morph_k=mk, open_iters=oi, close_iters=ci)
        key = f"k{mk}_o{oi}_c{ci}"
        try:
            eng.edges(masks, ec, out=edges)
        except omni_b200.OmniError as e:
            out[key] = {"supported": False, "error": str(e)[:120]}
            continue
        for _ in range(warmup):
            eng.edges(masks, ec, out=edges)
        torch.cuda.synchronize()
        ts = []
        for _ in range(steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); eng.edges(masks, ec, out=edges); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        v = edges.view(-1).view(torch.int64)
        i = torch.arange(v.numel(), device="cuda", dtype=torch.int64) % 1000003 + 1
        out[key] = {"supported": True, "ms_median": round(statistics.median(ts), 4), "ms_min": round(min(ts), 4),
                    "edge_csum": int((v * i).sum().item())}
    print(json.dumps({"lib": os.path.basename(omni_b200.LIB_PATH), "cases": out}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", default=os.path.join(PKG, "lib", "libomni_base.so"))
    ap.add_argument("--new", default=os.path.join(PKG, "lib", "libomni_b200.so"))
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true")
    a = ap.parse_args()
    if a.worker:
        worker(a.steps, a.warmup)
        return
    import torch
    card = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:          # the record still names the card through torch
        q = f"nvidia-smi unavailable: {e}"
    runs = {"base": [], "new": []}
    for _ in range(a.rounds):
        for tag, lib in (("base", a.base), ("new", a.new)):
            env = dict(os.environ, OMNI_B200_LIB=lib)
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(a.steps), "--warmup", str(a.warmup)],
                               env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            if r.returncode != 0 or not line:
                raise RuntimeError(f"{tag} worker failed:\n{r.stdout[-3000:]}")
            runs[tag].append(json.loads(line[-1])["cases"])
    summary = {}
    for mk, oi, ci in CASES:
        key = f"k{mk}_o{oi}_c{ci}"
        row = {}
        for tag in ("base", "new"):
            rs = [c[key] for c in runs[tag]]
            if all(x["supported"] for x in rs):
                row[f"{tag}_ms_median"] = round(statistics.median(x["ms_median"] for x in rs), 4)
                row[f"{tag}_ms_per_round"] = [x["ms_median"] for x in rs]
            else:
                row[f"{tag}_ms_median"] = None
                row[f"{tag}_error"] = rs[0].get("error")
        b, n = runs["base"][0][key], runs["new"][0][key]
        row["outputs_equal"] = (b["edge_csum"] == n["edge_csum"]) if b["supported"] and n["supported"] else None
        if row["base_ms_median"] and row["new_ms_median"]:
            row["speedup"] = round(row["base_ms_median"] / row["new_ms_median"], 2)
        summary[key] = row
    rec = {"probe": "morph_probe", "workload": "omni_edges 4096x4096, K=16 synth masks, edge_kernel_size 3, 50/150",
           "card": card, "nvidia_smi": q, "rounds": a.rounds, "steps": a.steps, "warmup": a.warmup,
           "libs": {"base": os.path.basename(a.base), "new": os.path.basename(a.new)}, "cases": summary}
    s = json.dumps(rec)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
