"""Summarise `ncu --set full` captures (.ncu-rep) into profiles/<name>.json: per captured launch the duration,
DRAM bytes, DRAM / L2 / tensor-pipe utilisation, occupancy, registers, shared memory; per kernel class the
average DRAM traffic per launch (the `roofline.traffic` figure bench.py reads from profiles/r2_ncu_summary.json).

    python tools/ncu_summary.py --out profiles/r2_ncu_summary.json flushed=profiles/r2_ncu_full_flushed_raw.csv live=profiles/r2_ncu_full_live_raw.csv
"""
import argparse
import csv
import io
import json
import subprocess
import sys

CLASS_OF = [("gemm_img", "linear"), ("gemm_chain", "linear"), ("token_fused", "token_fused"), ("sig_attention", "sig_attention"),
            ("match_tc", "match_tc"), ("match_tail", "match_tail"), ("match_exact", "match_exact"), ("desc_tiles", "desc_tiles")]

WANT = {
    "gpu__time_duration.sum": "duration_us",
    "dram__bytes_read.sum": "dram_read_bytes",
    "dram__bytes_write.sum": "dram_write_bytes",
    "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed": "dram_throughput_pct",
    "lts__throughput.avg.pct_of_peak_sustained_elapsed": "l2_throughput_pct",
    "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active": "tensor_pipe_active_pct",
    "sm__pipe_tensor_subpipe_hmma_cycles_active.avg.pct_of_peak_sustained_active": "tensor_pipe_hmma_active_pct",
    "sm__warps_active.avg.pct_of_peak_sustained_active": "warps_active_pct",
    "sm__throughput.avg.pct_of_peak_sustained_elapsed": "sm_throughput_pct",
    "launch__registers_per_thread": "registers",
    "launch__shared_mem_per_block_dynamic": "dyn_smem_bytes",
    "lts__t_sector_hit_rate.pct": "l2_hit_pct",
    "smsp__warp_issue_stalled_long_scoreboard_per_warp_active.pct": "stall_long_scoreboard_pct",
    "smsp__average_warps_issue_stalled_long_scoreboard_per_issue_active.ratio": "stall_long_scoreboard_per_issue",
    "smsp__average_warps_issue_stalled_short_scoreboard_per_issue_active.ratio": "stall_short_scoreboard_per_issue",
    "smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio": "stall_barrier_per_issue",
    "smsp__average_warps_issue_stalled_wait_per_issue_active.ratio": "stall_wait_per_issue",
}
UNIT_SCALE = {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12, "byte": 1.0, "ms": 1e3, "us": 1.0, "ns": 1e-3, "s": 1e6,
              "msecond": 1e3, "usecond": 1.0, "nsecond": 1e-3, "second": 1e6}


def read_report(path):
    if path.endswith(".csv"):     # already exported on the GPU box: ncu -i x.ncu-rep --page raw --csv
        raw = open(path).read()
    else:
        raw = subprocess.run(["ncu", "-i", path, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(raw)))
    hdr, units, data = rows[0], rows[1], rows[2:]
    col = {}
    for i, h in enumerate(hdr):
        base = h.split(".", 2)[-1] if h.count(".") >= 2 and h.split(".")[1] in ("TriageCompute",) else h
        for want in WANT:
            if h == want or h.endswith("." + want) or base == want:
                col.setdefault(want, i)
    out = []
    name_i, grid_i, block_i = hdr.index("Kernel Name"), hdr.index("Grid Size"), hdr.index("Block Size")
    for r in data:
        if len(r) < len(hdr):
            continue
        e = {"kernel": r[name_i].replace("void ", "").split("(")[0].replace("ltr::", ""), "grid": r[grid_i], "block": r[block_i]}
        for want, key in WANT.items():
            if want in col and r[col[want]] not in ("", "no data", "n/a"):
                try:
                    v = float(r[col[want]].replace(",", ""))
                except ValueError:
                    continue
                u = units[col[want]]
                if key.endswith("_bytes") or key == "duration_us":
                    v *= UNIT_SCALE.get(u, 1.0)
                e[key] = v
        out.append(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--note", default="")
    ap.add_argument("reports", nargs="+", help="tag=path.ncu-rep; the tag named 'flushed' feeds traffic_bytes_per_launch")
    args = ap.parse_args()
    res = {"note": args.note, "captures": {}}
    for spec in args.reports:
        tag, path = spec.split("=", 1)
        res["captures"][tag] = {"report": path, "launches": read_report(path)}
    src = res["captures"].get("flushed") or next(iter(res["captures"].values()))
    traffic, live = {}, {}
    for frag, cls in CLASS_OF:
        rows = [l for l in src["launches"] if frag in l["kernel"] and "dram_read_bytes" in l]
        if rows:
            tot = traffic.get(cls, [0.0, 0])
            traffic[cls] = [tot[0] + sum(l["dram_read_bytes"] + l.get("dram_write_bytes", 0.0) for l in rows), tot[1] + len(rows)]
    res["traffic_bytes_per_launch"] = {k: v[0] / v[1] for k, v in traffic.items()}
    res["traffic_source"] = "dram__bytes_read.sum + dram__bytes_write.sum, average over the captured launches of the class; " \
                            "ncu default cache control (L2 flushed before every replay): an upper bound of the live traffic"
    if "live" in res["captures"]:
        for frag, cls in CLASS_OF:
            rows = [l for l in res["captures"]["live"]["launches"] if frag in l["kernel"] and "dram_read_bytes" in l]
            if rows:
                tot = live.get(cls, [0.0, 0])
                live[cls] = [tot[0] + sum(l["dram_read_bytes"] + l.get("dram_write_bytes", 0.0) for l in rows), tot[1] + len(rows)]
        res["traffic_bytes_per_launch_cache_control_none"] = {k: v[0] / v[1] for k, v in live.items()}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"traffic_bytes_per_launch": res["traffic_bytes_per_launch"],
                      "live": res.get("traffic_bytes_per_launch_cache_control_none")}))
    for tag, c in res["captures"].items():
        print(tag)
        for l in c["launches"]:
            print("  %-28s %-14s %8.1f us  dramR %7.1f MB  dramW %6.1f MB  dram%% %5.1f  L2%% %5.1f  tensor%% %5.1f  warps%% %5.1f  regs %3d" % (
                l["kernel"][:28], l["grid"], l.get("duration_us", 0), l.get("dram_read_bytes", 0) / 1e6, l.get("dram_write_bytes", 0) / 1e6,
                l.get("dram_throughput_pct", 0), l.get("l2_throughput_pct", 0), l.get("tensor_pipe_active_pct", 0),
                l.get("warps_active_pct", 0), int(l.get("registers", 0))))


if __name__ == "__main__":
    main()
