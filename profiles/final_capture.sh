#!/bin/bash
# Everything the round's profile set is made of, in one GPU-box call (plain runs first, ncu afterwards):
#   bash profiles/final_capture.sh <tag>      -> gpurun_out/<tag>_*
set -u
TAG=${1:-r02z}
OUT=gpurun_out
(timeout 1200 python -m pytest tests -m gpu -x -q --timeout 400 2>&1 | tail -4) > $OUT/${TAG}_tests.log; cat $OUT/${TAG}_tests.log
timeout 600 python bench.py --steps 40 --warmup 3 > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err; echo "bench rc=$?"
timeout 400 python bench.py --steps 40 --warmup 3 --serial-steps --no-dropin > $OUT/${TAG}_bench_serial_steps.json 2> /dev/null
timeout 400 python bench.py --workload config4 --steps 20 --warmup 3 > $OUT/${TAG}_bench_c4.json 2> $OUT/${TAG}_bench_c4.err; echo "config4 rc=$?"
for HM in 2 5; do timeout 300 python bench.py --workload config4 --hough-method $HM --steps 20 --warmup 3 --no-verify > $OUT/${TAG}_bench_c4_hm$HM.json 2> /dev/null; done
timeout 900 python bench.py --workload config5 > $OUT/${TAG}_bench_c5.json 2> $OUT/${TAG}_bench_c5.err; echo "config5 rc=$?"
timeout 300 python bench.py --impl reference --steps 2 --warmup 1 > $OUT/${TAG}_bench_reference.json 2> /dev/null
timeout 300 python profiles/ktiming.py 64 > $OUT/${TAG}_ktiming.txt 2>&1
bash profiles/inst_list.sh $TAG > /dev/null 2>&1; rm -f $OUT/inst_$TAG.csv
bash profiles/ncu_kernel.sh ${TAG}_top "k_nms_march|k_morph_march|k_hough_vote|k_ccl_band|k_prep|k_rects_warp" 12 14 > /dev/null 2>&1
ls -la $OUT | grep $TAG
