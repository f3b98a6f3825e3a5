#!/bin/bash
# Round profile capture (run on the GPU box through gpurun): plain run first, then the ncu launch list of the
# same command, then one --set full capture of the top kernels.  usage: bash profiles/capture.sh <tag> [batch]
set -u
TAG=${1:-r01x}; B=${2:-64}
OUT=gpurun_out
CMD="python bench.py --profile --batch $B --steps 2 --warmup 3"
$CMD > $OUT/plain_$TAG.json 2> $OUT/plain_$TAG.err || { echo "plain run failed"; exit 1; }
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $OUT/launches_$TAG.csv $CMD > $OUT/ncu_l_$TAG.log 2>&1
echo "launch list rc=$?"
ncu --set full --clock-control none --import-source on \
    -k regex:"k_prep|k_morph_march|k_nms_march|k_ccl_band|k_rects_warp|k_hough_vote|k_ccl_stats" -s 132 -c 33 \
    -o $OUT/prof_$TAG -f $CMD > $OUT/ncu_f_$TAG.log 2>&1
echo "full capture rc=$?"
# the small kernels of the CCL / geometry / Hough tail (source-level data for the next round of tuning)
ncu --set full --clock-control none --import-source on \
    -k regex:"k_ccl_merge|k_ccl_alloc|k_ccl_extremes|k_fill_boxes|k_hough_compact|k_hough_peaks|k_hough_topk|k_star_mask" -s 100 -c 40 \
    -o $OUT/prof_${TAG}_small -f $CMD > $OUT/ncu_s_$TAG.log 2>&1
echo "small-kernel capture rc=$?"
ncu -i $OUT/prof_$TAG.ncu-rep --page raw --csv > $OUT/prof_${TAG}_raw.csv 2>/dev/null
ls -la $OUT/prof_$TAG.ncu-rep $OUT/prof_${TAG}_raw.csv
