#!/bin/bash
# Round profile capture (run under gpurun, ONE GPU): profile_round.sh <tag> <part>, part = bench | dense | stochvol.
# Outputs land in gpurun_out/ (kept small: .ncu-rep files are exported to CSV on the box and deleted) and are summarised
# into profiles/ by scripts/summarise_profiles.py.  Every ncu invocation runs under `timeout`; only the application
# process is profiled (bench.py spawns nvidia-smi and, for the CPU baseline, a process pool: profiling those children
# crashed ncu and left the counter library unusable for the next capture).
R=${1:-r1}
PART=${2:-bench}
O=gpurun_out
T=/tmp/ncu_$R
mkdir -p $T $O
NCU="ncu --target-processes application-only --clock-control none"
cap() {  # name kernel-regex skip script args...
  local name=$1 rx=$2 skip=$3; shift 3
  timeout -k 10 300 $NCU --set full --import-source on -k regex:$rx -s $skip -c 1 -o $T/$name -f python "$@" > $O/${R}_$name.log 2>&1
  echo "cap $name rc=$?"
  [ -f $T/$name.ncu-rep ] || return
  ncu -i $T/$name.ncu-rep --page raw --csv > $O/${R}_${name}_raw.csv 2>/dev/null
  ncu -i $T/$name.ncu-rep --page source --csv 2>/dev/null | gzip -9 > $O/${R}_${name}_src.csv.gz
  rm -f $T/$name.ncu-rep
}
if [ "$PART" = bench ]; then
  cap nuts nuts_warp_kernel 0 scripts/ncu_target_radon.py
  timeout -k 10 300 $NCU --metrics gpu__time_duration.sum -c 600 --csv --log-file $O/${R}_launches.csv python bench.py --steps 2 --warmup 1 --no-cpu-baseline > $O/${R}_launches_bench.log 2>&1
  echo "launch list rc=$?"
elif [ "$PART" = tc ]; then
  timeout -k 10 200 $NCU --metrics gpu__time_duration.sum -c 300 --csv --log-file $O/${R}_launches_logistic_tc.csv python scripts/ncu_target3.py logistic_tc 4 2 > $O/${R}_launches_logistic_tc.log 2>&1
  timeout -k 10 200 $NCU --metrics gpu__time_duration.sum -c 300 --csv --log-file $O/${R}_launches_mvgauss_tc.csv python scripts/ncu_target3.py mvgauss_tc 4 2 > $O/${R}_launches_mvgauss_tc.log 2>&1
  cap gemm_tc gemm_tc_kernel 4 scripts/ncu_target3.py mvgauss_tc 2 1
elif [ "$PART" = tc2 ]; then  # the tensor-core logistic pass only
  timeout -k 10 200 $NCU --metrics gpu__time_duration.sum -c 300 --csv --log-file $O/${R}_launches_logistic_tc.csv python scripts/ncu_target3.py logistic_tc 4 2 > $O/${R}_launches_logistic_tc.log 2>&1
  cap logistic_tc logistic_tc2_kernel 2 scripts/ncu_target3.py logistic_tc 2 1
elif [ "$PART" = stochvol ]; then
  cap stochvol nuts_warp_kernel 0 scripts/ncu_target_stochvol.py
else
  timeout -k 10 200 $NCU --metrics gpu__time_duration.sum -c 300 --csv --log-file $O/${R}_launches_logistic.csv python scripts/ncu_target3.py logistic 4 2 > $O/${R}_launches_logistic.log 2>&1
  cap logistic logistic_fused_kernel 2 scripts/ncu_target3.py logistic 2 1
  timeout -k 10 200 $NCU --metrics gpu__time_duration.sum -c 300 --csv --log-file $O/${R}_launches_mvgauss.csv python scripts/ncu_target3.py mvgauss 4 2 > $O/${R}_launches_mvgauss.log 2>&1
  cap gemm gemm_nt_dmma_kernel 4 scripts/ncu_target3.py mvgauss 2 1
fi
for f in $O/${R}_*.log; do echo "== $f"; tail -n 2 $f | cut -c1-300; done
du -sh $O
