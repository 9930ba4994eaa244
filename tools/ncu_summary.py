"""Summarise ncu output into tracked text files under profiles/.

  python tools/ncu_summary.py launches launches_step.csv profiles/r01_launch_shares.txt
  python tools/ncu_summary.py full prof_hot.ncu-rep profiles/r01_ncu_hot.txt [profiles/ncu_traffic.json]

launches_step.csv is ncu's --csv log of gpu__time_duration.sum per launch, prof_hot.ncu-rep a --set full report, both of a run
of tools/probe.py.
"""
import collections, csv, json, re, subprocess, sys

def launches(src, dst):
    lines = [l for l in open(src) if not l.startswith("==")]
    agg = collections.defaultdict(lambda: [0, 0.0]); tot = 0.0
    for row in csv.DictReader(lines):
        if row.get("Metric Name") != "gpu__time_duration.sum":
            continue
        name = row["Kernel Name"]
        m = re.search(r"ps_for_kernel<.*?ps::(\w+)\(", name)
        name = ("ps_for:" + m.group(1)) if m else name.split("(")[0]
        v = float(row["Metric Value"].replace(",", "")); u = row["Metric Unit"]
        v = v / 1e6 if u in ("nsecond", "ns") else v / 1e3 if u in ("usecond", "us") else v
        agg[name][0] += 1; agg[name][1] += v; tot += v
    with open(dst, "w") as f:
        f.write(f"# ncu --metrics gpu__time_duration.sum --clock-control none: one full step (cold-cache, serialised; compare SHARES)\n# source: {src}\n")
        f.write(f"total {tot:.3f} ms over {sum(c for c, _ in agg.values())} launches\n")
        for k, (c, t) in sorted(agg.items(), key=lambda x: -x[1][1]):
            f.write("%-60s n=%5d %10.3f ms %5.1f%%  avg %.4f ms\n" % (k[:60], c, t, 100 * t / tot, t / c))
    print(open(dst).read()[:3000])

WANT = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
        "dram__throughput.avg.pct_of_peak_sustained_elapsed", "launch__registers_per_thread", "launch__grid_size", "launch__block_size",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
        "l1tex__t_sector_hit_rate.pct", "lts__t_sector_hit_rate.pct", "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum", "smsp__inst_executed.sum",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "sm__inst_executed_pipe_fp64.sum"]

def full(src, dst, traffic_json=None):
    out = subprocess.run(["ncu", "-i", src, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(out.splitlines())); hdr, units = rows[0], rows[1]; idx = {h: i for i, h in enumerate(hdr)}
    traffic = {}
    with open(dst, "w") as f:
        f.write(f"# ncu --set full --clock-control none --import-source on; source: {src}\n")
        for r in rows[2:]:
            kn = r[idx["Kernel Name"]].split("(")[0]
            f.write(f"---- {kn}\n")
            for w in WANT:
                if w in idx:
                    f.write("   %-72s %s %s\n" % (w, r[idx[w]], units[idx[w]]))
            def gb(name):
                v = float(r[idx[name]].replace(",", "")); u = units[idx[name]]
                return v * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(u, 1)
            traffic[kn] = gb("dram__bytes_read.sum") + gb("dram__bytes_write.sum")
            f.write("   %-72s %.6f GB\n" % ("traffic = dram read + write per launch", traffic[kn] / 1e9))
    if traffic_json:
        json.dump(traffic, open(traffic_json, "w"), indent=1)
    print(open(dst).read())

if __name__ == "__main__":
    if sys.argv[1] == "launches": launches(sys.argv[2], sys.argv[3])
    else: full(*sys.argv[2:])
