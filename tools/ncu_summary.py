#!/usr/bin/env python3
"""Summarise an `ncu --set full` report into profiles/:  python tools/ncu_summary.py REPORT.ncu-rep OUT.json [--traffic config2]

Writes one record per captured launch (duration, DRAM bytes, instructions, IPC, occupancy, registers, grid) and, with
--traffic WORKLOAD, refreshes profiles/traffic.json (dram read + write bytes per launch, keyed by the names bench.py uses)."""
import csv
import json
import os
import subprocess
import sys

KEYS = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum", "smsp__inst_executed.sum",
        "sm__inst_executed.avg.per_cycle_elapsed", "sm__warps_active.avg.pct_of_peak_sustained_active",
        "smsp__issue_active.avg.pct_of_peak_sustained_active", "launch__registers_per_thread", "launch__grid_size",
        "launch__block_size", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__t_sector_hit_rate.pct", "lts__t_sector_hit_rate.pct"]
BENCH_NAME = {"fk_assign_rgbcell": "assign_bits", "fk_assign_bits": "assign_bits", "fk_assign_slices": "assign_bits", "fk_morph": "morph_bits",
              "fk_morph_lab": "morph_bits", "fk_label_open": "label_open", "fk_open_morph": "morph_bits", "fk_build_tables3": "build_tables",
              "fk_edges3_simd": "edges3_bits", "fk_hysteresis": "hysteresis_bits", "fk_edge_runs": "edge_runs", "fk_thin": "thin_zhangsuen"}
UNIT = {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}


def main():
    rep, out = sys.argv[1], sys.argv[2]
    txt = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], stdout=subprocess.PIPE, text=True, check=True).stdout
    rows = list(csv.reader(txt.splitlines()))
    hdr, units = rows[0], rows[1]
    idx = {n: i for i, n in enumerate(hdr)}
    recs, traffic = [], {}
    for r in rows[2:]:
        name = r[idx["Kernel Name"]]
        short = name.split("(")[0].replace("void ", "").strip()
        rec = {"kernel": short}
        for k in KEYS:
            if k in idx:
                rec[k] = f"{r[idx[k]]} {units[idx[k]]}".strip()
        recs.append(rec)
        base = short.split("<")[0]
        if base in BENCH_NAME:
            b = sum(float(r[idx[k]].replace(",", "")) * UNIT.get(units[idx[k]], 1.0) for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
            traffic[BENCH_NAME[base]] = int(b)
    json.dump(recs, open(out, "w"), indent=1)
    print("wrote", out, len(recs), "launches")
    if "--traffic" in sys.argv:
        wl = sys.argv[sys.argv.index("--traffic") + 1]
        tp = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "traffic.json")
        t = json.load(open(tp)) if os.path.exists(tp) else {}
        t[wl] = traffic
        t["_source"] = f"ncu --set full, {os.path.basename(out)} (dram__bytes_read.sum + dram__bytes_write.sum per launch)"
        json.dump(t, open(tp, "w"), indent=1)
        print("updated", tp, traffic)


if __name__ == "__main__":
    main()
