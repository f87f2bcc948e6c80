"""Turn the captures of tools/profile_round.sh (gpurun_out/) into the committed summaries under profiles/:
launch-list summary, key ncu metrics per kernel, and profiles/traffic.json (DRAM bytes per launch, read by bench.py)."""
import csv, json, os, shutil, subprocess, sys
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = sys.argv[1] if len(sys.argv) > 1 else "r2"
G, P = os.path.join(REPO, "gpurun_out"), os.path.join(REPO, "profiles")


def run(*cmd):
    return subprocess.run(cmd, capture_output=True, text=True).stdout


for name in (f"{R}_bench_launches.csv", f"{R}_stage_profile.log", f"{R}_nms_phases.log",
             f"{R}_msroialign.log", f"{R}_roi_bwd_probe.log"):
    if os.path.exists(os.path.join(G, name)):
        shutil.copy(os.path.join(G, name), os.path.join(P, name))
open(os.path.join(P, f"{R}_bench_launches_summary.txt"), "w").write(
    run(sys.executable, os.path.join(REPO, "tools", "launch_summary.py"), os.path.join(G, f"{R}_bench_launches.csv")))
lines = []
for w in ("all", "reference", "rpn", "train", "infer", "joint", "all_n2", "all_n4", "all_n8"):   # the multi-GPU lines come from separate gpurun --gpus N calls
    f = os.path.join(G, f"{R}_bench_{w}.json")
    if os.path.exists(f):
        js = [l for l in open(f).read().splitlines() if l.startswith("{")]   # (torchrun prints a banner on stdout)
        if js:
            lines.append(js[-1])
open(os.path.join(P, f"{R}_bench.json"), "w").write("\n".join(lines) + "\n")
traffic = {}
for tag in ("proposal", "roi"):
    rep = os.path.join(G, f"prof_{R}_{tag}.ncu-rep")
    if not os.path.exists(rep):
        continue
    open(os.path.join(P, f"{R}_{tag}_kernels_ncu.txt"), "w").write(
        run(sys.executable, os.path.join(REPO, "tools", "ncu_summary.py"), rep))
    rows = list(csv.reader(run("ncu", "-i", rep, "--page", "raw", "--csv").splitlines()))
    hdr, units = rows[0], rows[1]
    scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for r in rows[2:]:
        k = r[hdr.index("Kernel Name")].split("(")[0].split("<")[0].replace("void ", "").strip()
        rd, wr = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        traffic.setdefault(k, {"dram_bytes_read": float(r[rd].replace(",", "")) * scale[units[rd]],
                               "dram_bytes_write": float(r[wr].replace(",", "")) * scale[units[wr]],
                               "us_under_ncu": float(r[hdr.index("gpu__time_duration.sum")].replace(",", "")) *
                               {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}.get(units[hdr.index("gpu__time_duration.sum")], 1.0),
                               "inst_executed": float(r[hdr.index("smsp__inst_executed.sum")].replace(",", "")),
                               "source": f"profiles/{R}_{tag}_kernels_ncu.txt (ncu --set full, one launch, cold L2 state of the bench)"})
json.dump(traffic, open(os.path.join(P, "traffic.json"), "w"), indent=1)
print(json.dumps(traffic, indent=1))
