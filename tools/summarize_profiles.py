"""Turn gpurun_out/ ncu artefacts into tracked summaries under profiles/.
usage: python tools/summarize_profiles.py <round-tag>     (reads gpurun_out/launches_<tag>.csv, prof_*_<tag>.ncu-rep)"""
import collections
import csv
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tag = sys.argv[1] if len(sys.argv) > 1 else "r1"
G, P = os.path.join(ROOT, "gpurun_out"), os.path.join(ROOT, "profiles")
os.makedirs(P, exist_ok=True)

KEYS = ["gpu__time_duration.sum", "launch__grid_size", "launch__block_size", "launch__registers_per_thread",
        "launch__shared_mem_per_block_dynamic", "sm__cycles_elapsed.max", "sm__cycles_active.avg",
        "sm__pipe_tensor_cycles_active_realtime.avg.pct_of_peak_sustained_elapsed",
        "sm__pipe_tensor_subpipe_hmma_cycles_active_realtime.avg",
        "sm__inst_executed_pipe_tensor.sum", "sm__warps_active.avg.pct_of_peak_sustained_active",
        "dram__bytes_read.sum", "dram__bytes_write.sum", "dram__throughput.avg.pct_of_peak_sustained_elapsed",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "lts__t_bytes.sum",
        "lts__throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum",
        "smsp__inst_executed.sum", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__inst_executed.avg.per_cycle_elapsed", "smsp__cycles_active.avg",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed", "smsp__warp_issue_stalled_long_scoreboard_per_warp_active.pct",
        "l1tex__t_sector_hit_rate.pct", "lts__t_sector_hit_rate.pct"]


TENSOR_KEYS = ["sm__pipe_tensor_cycles_active_realtime.avg.pct_of_peak_sustained_elapsed",
               "sm__pipe_tensor_subpipe_hmma_cycles_active_realtime.avg",
               "sm__mem_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed",
               "sm__mem_tensor_cycles_active.avg.pct_of_peak_sustained_active"]


def launches():
    path = os.path.join(G, "launches_%s.csv" % tag)
    if not os.path.exists(path):
        return
    rows = [r for r in csv.reader(open(path)) if len(r) > 5]
    hi = [i for i, r in enumerate(rows) if "Kernel Name" in r][0]
    hdr = rows[hi]
    kn, mv, mn = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Name")
    agg = collections.OrderedDict()
    for r in rows[hi + 1:]:
        if r[mn] != "gpu__time_duration.sum":
            continue
        a = agg.setdefault(r[kn].split("(")[0], [0, 0.0])
        a[0] += 1
        a[1] += float(r[mv].replace(",", ""))
    tot = sum(v[1] for v in agg.values())
    with open(os.path.join(P, "%s_launches.md" % tag), "w") as f:
        f.write("# ncu launch list, round %s\n\n" % tag)
        f.write(open(os.path.join(G, "launches_%s.cmd" % tag)).read() if os.path.exists(os.path.join(G, "launches_%s.cmd" % tag)) else "")
        f.write("\n(C3 workload: 500 games, 50 sims/move, batch 8, two launches per round; per-launch times are cold-cache and\n"
                "serialised -- compare SHARES, not absolutes)\n\n")
        f.write("| kernel | launches | total us | avg us | share |\n|---|---:|---:|---:|---:|\n")
        for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write("| %s | %d | %.1f | %.2f | %.1f%% |\n" % (k, v[0], v[1] / 1e3, v[1] / 1e3 / v[0], 100 * v[1] / tot))
    print(open(os.path.join(P, "%s_launches.md" % tag)).read())


def full(name):
    rep = os.path.join(G, "prof_%s_%s.ncu-rep" % (name, tag))
    if not os.path.exists(rep):
        return
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(raw.splitlines()))
    hdr, units = rows[0], rows[1]
    with open(os.path.join(P, "%s_%s_full.md" % (tag, name)), "w") as f:
        f.write("# ncu --set full, %s kernel, round %s\n\n" % (name, tag))
        f.write("`ncu --set full --clock-control none --import-source on -k regex:<kernel> ...` (commands: tools/gpu_round2.sh)\n\n")
        seen = set()
        for r in rows[2:]:
            kname = r[hdr.index("Kernel Name")].split("(")[0]
            if name == "rules" and kname in seen:      # several timed repetitions per kernel: keep the first
                continue
            seen.add(kname)
            f.write("## launch id %s: %s grid %s block %s\n\n| metric | unit | value |\n|---|---|---:|\n" % (
                r[0], r[hdr.index("Kernel Name")].split("(")[0], r[hdr.index("Grid Size")], r[hdr.index("Block Size")]))
            for i, h in enumerate(hdr):
                if h in KEYS or any(h.endswith(k) for k in TENSOR_KEYS):
                    f.write("| %s | %s | %s |\n" % (h, units[i], r[i]))
            f.write("\n")
    print(open(os.path.join(P, "%s_%s_full.md" % (tag, name))).read()[:3000])


launches()
full("trunk2")     # trunk_auto_kernel -> trunk_tc2_body<2> (CTA pair per group, 2 tiles per CTA; batch of 345 positions)
full("trunkx3")    # trunk_x3_kernel (split-bf16: 3 MMAs per K-block; batch of 500 positions = groups of 5 + 2 per CTA pair)
full("trunkpp")    # trunk_auto_kernel, launch 200 of a 500-game cycle (~495 positions): trunk_pp_body<1> (two groups in
                   # flight, cta_group::2) + heads FC tail
full("heads")      # heads_fc_kernel (standalone form of the heads' FC layers; 500 positions, warm L2)
full("tree")
full("rules")      # step / legal / encode / gather_planes / playout kernels at 2^22 (2^20) states (tools/prof_rules.py 22)
