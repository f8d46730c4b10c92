"""Copy the evidence of one capture round (tools/ncu_capture.sh, run under gpurun) from gpurun_out/ into profiles/:
    python tools/make_profiles.py r02_v1
bench JSON lines (both arms), the ncu launch list, one summary row per `ncu --set full` capture (one .ncu-rep per hot kernel),
the DRAM-traffic table that bench.py echoes as roofline.traffic, and per-instruction stall tables of the captures that
carry source (--import-source on)."""
import csv
import json
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tag = sys.argv[1]
src, dst = os.path.join(ROOT, "gpurun_out"), os.path.join(ROOT, "profiles")
for a, b in (("bench.json", "bench.json"), ("bench_ref.json", "bench_reference_arm.json"), ("launches.csv", "launches.csv")):
    if os.path.isfile(os.path.join(src, a)):
        shutil.copy(os.path.join(src, a), os.path.join(dst, f"{tag}_{b}"))

KEEP = ["Kernel Name", "launch__grid_size", "launch__block_size", "launch__registers_per_thread", "gpu__time_duration.sum",
        "sm__cycles_elapsed.avg.per_second", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__pipe_tensor_subpipe_hmma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_active", "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__pipe_xu_cycles_active.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__inst_executed.sum",
        "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum", "l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed"]
STALLS = ["barrier", "branch_resolving", "long_scoreboard", "short_scoreboard", "math_pipe_throttle", "mio_throttle", "wait",
          "sleeping", "not_selected", "selected", "no_instructions", "lg_throttle", "dispatch_stall"]
# capture -> (what one launch is, rows, algorithmic bytes per launch)  [SURVEY 8d per-item figures x rows of the launch]
ALGO = {
    "encoder": ("enc_mlp_kernel, 1 Mi rows of 768-d items -> z [N, 32]", 1 << 20, (1 << 20) * (4 * 768 + 4 * 32)),
    "rq_encode": ("rq_fwd_tc_v11_kernel<0,0> ids only, 4 Mi rows D32 K256 L3", 1 << 22, (1 << 22) * (4 * 32 + 8 * 3)),
    "train_fwd": ("rq_fwd_tc_v11_kernel<rot,out> emb_out + loss + ids, 4 Mi rows", 1 << 22, (1 << 22) * (4 * 32 + 4 * 32 * 3 + 8 * 3 + 4)),
    "train_bwd": ("rq_bwd_smem_kernel<32,8,rot,train,3>, 4 Mi rows", 1 << 22, (1 << 22) * (4 * 32 + 8 * 3 + 4 * 32 * 3 + 4 + 4 * 32) + 4 * 3 * 256 * 32),
    "c4": ("large-codebook encode 65,536 x D64 x K4096 x L4", 65536, 65536 * (4 * 64 + 8 * 4) + 4 * 4096 * (4 * 64 + 32) * 4),
    "kmeans": ("kmeans_segsum_kernel<64>, 65,536 rows, K 4096", 65536, 65536 * (4 * 64 + 12) + 4096 * 65 * 4),
    "uniq": ("uniq_sorted_kernel, 65,536 rows of 3 ids + 32-d features (every row has a twin)", 65536, 65536 * (8 * 3 + 12 + 4 * 32)),
}
SCALE = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
summary, traffic = [], {}
for name, (what, rows_n, algo_bytes) in ALGO.items():
    rep = os.path.join(src, f"ncu_{name}.ncu-rep")
    if not os.path.isfile(rep):
        continue
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(raw.splitlines()))
    h, u, r = rows[0], rows[1], rows[2]
    get = lambda k: r[h.index(k)] if k in h else ""
    unit = lambda k: u[h.index(k)] if k in h else ""
    row = {"capture": name, "launch": what}
    for k in KEEP:
        row[k] = (get(k) + " " + unit(k)).strip()
    for s in STALLS:
        key = f"smsp__average_warps_issue_stalled_{s}_per_issue_active.ratio"
        row["stall_" + s] = get(key)
    summary.append(row)
    rd = float(get("dram__bytes_read.sum")) * SCALE[unit("dram__bytes_read.sum")]
    wr = float(get("dram__bytes_write.sum")) * SCALE[unit("dram__bytes_write.sum")]
    ms = float(get("gpu__time_duration.sum")) * {"ms": 1.0, "us": 1e-3, "ns": 1e-6, "s": 1e3}[unit("gpu__time_duration.sum")]
    traffic[name] = dict(launch=what, dram_bytes=int(rd + wr), dram_read=int(rd), dram_write=int(wr), algorithmic_bytes=int(algo_bytes),
                         ratio=round((rd + wr) / algo_bytes, 3), ncu_ms=round(ms, 4), sm_ghz_under_ncu=get("sm__cycles_elapsed.avg.per_second"))
    srcp = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv"], capture_output=True, text=True).stdout
    if srcp.count("\n") > 50:
        tmp = f"/tmp/{tag}_{name}.csv"
        open(tmp, "w").write(srcp)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ncu_stalls.py"), tmp, "40"], capture_output=True, text=True).stdout
        if out.strip():
            open(os.path.join(dst, f"{tag}_ncu_stalls_{name}.txt"), "w").write(out)
with open(os.path.join(dst, f"{tag}_ncu_full_summary.csv"), "w", newline="") as f:
    w = csv.DictWriter(f, fieldnames=list(summary[0].keys()))
    w.writeheader()
    w.writerows(summary)
# keys bench.py looks up
traffic["enc_mlp_kernel"] = traffic.get("encoder", {}).get("dram_bytes")
traffic["rq_fwd_tc_v11_kernel_encode"] = traffic.get("rq_encode", {}).get("dram_bytes")
traffic["source"] = f"profiles/{tag}_ncu_full_summary.csv (ncu --set full --clock-control none, one launch per kernel at the shape named)"
traffic["note"] = ("enc_mlp_kernel is captured at 1 Mi rows (the bench's chunk); rq_fwd_tc_v11_kernel at 4 Mi rows: bench.py scales its "
                   "per-launch traffic to the rows of the launch it times")
json.dump(traffic, open(os.path.join(dst, "r02_traffic.json"), "w"), indent=1)
print(json.dumps(traffic, indent=1))
