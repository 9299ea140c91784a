#!/bin/bash
# One ncu --set full capture per kernel family at the BASELINE sizes (tools/kernel_times.py launches them all); text details and the
# raw metric table of each capture go to gpurun_out/ncu_r2/ (copied to profiles/ by hand).  Run on the GPU box, after the same
# program exited 0 without ncu.
cd "$(dirname "$0")/.."
out=gpurun_out/ncu_r2
mkdir -p $out
timeout 300 python tools/kernel_times.py > $out/kernel_times_plain.log 2>&1 || { echo "kernel_times.py failed without ncu"; tail -5 $out/kernel_times_plain.log; exit 1; }
# launch list of the whole program (durations only)
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:^k_ --csv --log-file $out/launches_all_kernel_families.csv python tools/kernel_times.py > /dev/null 2>&1
for k in k_flag_raw k_emit_flagged k_segment_nms_bins k_gather_rows k_decode_dense k_decode_train k_decode_train_bwd k_filter_dense_rows k_target_objmask k_target_scatter k_loss_match k_loss_obj; do
  skip=1
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:^$k -s $skip -c 1 -o $out/$k python tools/kernel_times.py > $out/$k.log 2>&1
  if [ -f $out/$k.ncu-rep ]; then
    ncu -i $out/$k.ncu-rep --page details > $out/${k}_details.txt 2>/dev/null
    ncu -i $out/$k.ncu-rep --page raw --csv > $out/${k}_raw.csv 2>/dev/null
    grep -E "Duration|DRAM Throughput|Issue Slots Busy|Registers Per|Achieved Occupancy" $out/${k}_details.txt | head -6 | sed "s/^/$k: /"
    rm -f $out/$k.ncu-rep
  else
    echo "$k: no report"; tail -3 $out/$k.log
  fi
done
YL_FLAG=tma timeout 600 ncu --set full --clock-control none --import-source on -k regex:^k_flag_tma -s 1 -c 1 -o $out/k_flag_tma python tools/step_probe.py > $out/k_flag_tma.log 2>&1
ncu -i $out/k_flag_tma.ncu-rep --page details > $out/k_flag_tma_details.txt 2>/dev/null
ncu -i $out/k_flag_tma.ncu-rep --page raw --csv > $out/k_flag_tma_raw.csv 2>/dev/null
rm -f $out/k_flag_tma.ncu-rep
# step launch list of the default chain
N=3 timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:^k_ -c 40 --csv --log-file $out/launches_step.csv python tools/step_probe.py > /dev/null 2>&1
ls -la $out | head -50
