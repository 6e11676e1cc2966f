#!/bin/bash
# Round-2 evidence capture on the GPU box (one B200): launch list of the bench command + `ncu --set full` of every shipped hot kernel.
# Usage: bash tools/r02_capture.sh [steps]   steps = any of: bench frame ops src   (default: all)
# Outputs land in gpurun_out/ (scratch, <= 64 MiB per call: the whole-frame reports are exported to raw CSV on the box, only the
# chain / attention / VFE / SIR single-launch reports travel as .ncu-rep with source); tools/ncu_summary.py condenses them into profiles/r02_*.
STEPS="${*:-bench frame ops src}"
O=gpurun_out
T=/tmp/r02
mkdir -p $O $T
NCU="ncu --clock-control none"
for s in $STEPS; do
case $s in
bench)
  # launch list (durations + DRAM bytes) of the bench command itself: the kernels of its first timed window (4 frames; the engines'
  # construction warm-ups run on empty buffers and are excluded by the profiler range bench.py opens under SSTB200_NCU_RANGE=1)
  SSTB200_NCU_RANGE=1 timeout 600 $NCU --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum \
      --profile-from-start off --csv --log-file $O/r02_launches_bench.csv \
      python bench.py --steps 4 --warmup 3 --no-train --no-fp32 --no-cpu-baseline > $O/r02_launches_bench.log 2>&1 ;;
frame)
  # one warm frame of the flagship pipeline, every kernel, full set -> raw CSV
  timeout 900 $NCU --set full --profile-from-start off -o $T/frame -f python tools/frame_kernels.py > $O/r02_frame_full.log 2>&1
  ncu -i $T/frame.ncu-rep --page raw --csv > $O/r02_frame_full_raw.csv ;;
ops)
  # FSD SIR (config 3) and the scatter ops (config 2 shape), warm passes -> raw CSV
  timeout 600 $NCU --set full --profile-from-start off -o $T/sir -f python tools/sir_kernels.py > $O/r02_sir_full.log 2>&1
  ncu -i $T/sir.ncu-rep --page raw --csv > $O/r02_sir_full_raw.csv
  timeout 600 $NCU --set full --profile-from-start off -o $T/scatter -f python tools/scatter_kernels.py > $O/r02_scatter_full.log 2>&1
  ncu -i $T/scatter.ncu-rep --page raw --csv > $O/r02_scatter_full_raw.csv
  timeout 600 $NCU --set full --import-source on --profile-from-start off -k regex:vfe_l1_umma_kernel -c 1 -o $O/r02_vfe_l1 -f python tools/frame_kernels.py > /dev/null 2>&1
  timeout 600 $NCU --set full --import-source on --profile-from-start off -k regex:'sir_[ab]_kernel' -c 2 -o $O/r02_sir_ab -f python tools/sir_kernels.py > /dev/null 2>&1 ;;
src)
  # single launches with source (mid-stack layer): chain, attention
  timeout 600 $NCU --set full --import-source on --profile-from-start off -k regex:sra_chain2_kernel -s 5 -c 1 -o $O/r02_chain2 -f python tools/frame_kernels.py > /dev/null 2>&1
  timeout 600 $NCU --set full --import-source on --profile-from-start off -k regex:win_attn_batch_kernel -s 5 -c 1 -o $O/r02_attn -f python tools/frame_kernels.py > /dev/null 2>&1 ;;
esac
done
ls -la $O/r02_*
