#!/bin/bash
# tools/ncu_capture.sh [TAG]: the round's evidence run on the GPU box (under gpurun, one GPU).  Everything lands in
# gpurun_out/; tools/make_profiles.py TAG then copies the summaries into profiles/.
#   1. python bench.py, python bench.py --impl reference      (never under a profiler)
#   2. ncu launch list of a short bench.py run                  (per-launch durations, cold caches, serialised)
#   3. one `ncu --set full` capture per hot kernel at its bench shape (tools/run_kernels_once.py)
set -u
cd "$(dirname "$0")/.."
out=gpurun_out
mkdir -p $out
python bench.py > $out/bench.json 2> $out/bench.err; echo "bench rc=$?"
python bench.py --impl reference > $out/bench_ref.json 2> $out/bench_ref.err; echo "reference arm rc=$?"
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $out/launches.csv \
    python bench.py --steps 2 --warmup 1 --no-sweep > $out/ncu_list.log 2>&1; echo "launch list rc=$?"
cap() {  # name, workload of run_kernels_once.py, kernel regex, launches to skip, extra flags
  timeout 600 ncu --set full --clock-control none $5 -k "regex:$3" -s $4 -c 1 -f -o $out/ncu_$1 \
      python tools/run_kernels_once.py $2 > $out/ncu_$1.log 2>&1; echo "ncu $1 rc=$?"
}
cap encoder   encoder 'enc_mlp_kernel'       1 "--import-source on"
cap rq_encode rq      'rq_fwd_tc_v11_kernel' 1 "--import-source on"
cap train_fwd train   'rq_fwd_tc_v11_kernel' 1 ""
cap train_bwd train   'rq_bwd_smem_kernel'   1 "--import-source on"
cap c4        c4      'rq_fwd_tc'            1 "--import-source on"
cap kmeans    aux     'kmeans_segsum_kernel' 0 ""
cap uniq      aux     'uniq_sorted_kernel'   0 ""
ls -la $out/*.ncu-rep
